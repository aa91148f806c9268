"""
Thin numpy wrapper over the device seam (include/plf.h).  Every method is a
direct call into libarbplf_b200.so; nothing is computed in Python.
"""
import ctypes

import numpy as np

from . import _lib

ROOT_NONE, ROOT_UNIFORM, ROOT_EQUILIBRIUM, ROOT_CUSTOM = range(4)
KIND_DWELL, KIND_TRANS = 0, 1
PATH_AUTO, PATH_GENERIC, PATH_FUSED4 = 0, 1, 2


CODES_PACKED4 = 0       # include/plf.h: PLF_CODES_PACKED4


def pack4(codes, out=None):
    """[S][N] codes below 16 -> [S][(N + 1) // 2] bytes, node 2j in the low and node 2j + 1 in the high nibble."""
    codes = np.asarray(codes)
    S, N = codes.shape
    if codes.size and int(codes.max()) > 15:
        raise ValueError("pack4: codes must be below 16")
    M = (N + 1) // 2
    if out is None:
        out = np.empty((S, M), dtype=np.uint8)
    np.copyto(out[:, :N // 2], codes[:, 1:2 * (N // 2):2].astype(np.uint8) << 4)
    out[:, :N // 2] |= codes[:, 0:2 * (N // 2):2].astype(np.uint8)
    if N % 2:
        out[:, M - 1] = codes[:, N - 1]
    return out


class EngineError(RuntimeError):
    pass


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _f64(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


class Engine:
    def __init__(self, device=0):
        self._lib = _lib.load()
        self._h = ctypes.c_void_p()
        if self._lib.plf_create(ctypes.byref(self._h), device) != 0:
            raise EngineError("plf_create failed: no usable CUDA device (there is no CPU path)")
        self.N = self.E = self.n = self.C = 0
        self.S = 0

    def close(self):
        if self._h:
            self._lib.plf_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise EngineError(self._lib.plf_last_error(self._h).decode())

    def set_path(self, path):
        self._ck(self._lib.plf_set_path(self._h, path))

    def set_tree(self, indptr, indices, preorder):
        indptr = np.ascontiguousarray(indptr, dtype=np.int32)
        indices = np.ascontiguousarray(indices, dtype=np.int32)
        preorder = np.ascontiguousarray(preorder, dtype=np.int32)
        self.N = len(preorder)
        self.E = self.N - 1
        self._ck(self._lib.plf_set_tree(self._h, self.N, _ptr(indptr), _ptr(indices), _ptr(preorder)))

    def set_model(self, q_hi, q_lo, edge_rates, cat_rates, cat_prior, root_mode, root_vec=None):
        q_hi = _f64(q_hi)
        q_lo = _f64(q_lo)
        self.n = q_hi.shape[0]
        cat_rates = _f64(cat_rates)
        self.C = len(cat_rates)
        self._ck(self._lib.plf_set_model(self._h, self.n, self.C, _ptr(q_hi), _ptr(q_lo), _ptr(_f64(edge_rates)),
                                         _ptr(cat_rates), _ptr(_f64(cat_prior)), root_mode, _ptr(_f64(root_vec))))

    def set_edge_rates(self, edge_rates):
        self._ck(self._lib.plf_set_edge_rates(self._h, _ptr(_f64(edge_rates))))

    def set_data(self, defs, codes):
        """defs [K][n] float64; codes [S][N] uint8 or int32."""
        defs = _f64(defs)
        if codes.dtype == np.uint8:
            cb = 1
        else:
            codes = np.ascontiguousarray(codes, dtype=np.int32)
            cb = 4
        codes = np.ascontiguousarray(codes)
        self.S = codes.shape[0]
        self._ck(self._lib.plf_set_data(self._h, self.S, defs.shape[0], _ptr(defs), _ptr(codes), cb))

    def set_data_packed(self, defs, packed, weights=None, asynchronous=False):
        """Codes as PLF_CODES_PACKED4 rows (pack4): half the upload of uint8 codes."""
        defs = _f64(defs)
        packed = np.ascontiguousarray(packed, dtype=np.uint8)
        self.S = packed.shape[0]
        if asynchronous:
            weights = None if weights is None else _f64(weights)
            self._pending_host = (packed, weights)
            self._ck(self._lib.plf_set_data_async(self._h, self.S, defs.shape[0], _ptr(defs), _ptr(packed), CODES_PACKED4,
                                                  _ptr(weights)))
        else:
            self._ck(self._lib.plf_set_data(self._h, self.S, defs.shape[0], _ptr(defs), _ptr(packed), CODES_PACKED4))
            if weights is not None:
                self.set_site_weights(weights)

    def set_data_ptr(self, defs, codes_ptr, S, code_bytes=1):
        defs = _f64(defs)
        self.S = S
        self._ck(self._lib.plf_set_data(self._h, S, defs.shape[0], _ptr(defs), ctypes.c_void_p(codes_ptr), code_bytes))

    def set_data_async(self, defs, codes, weights=None):
        """plf_set_data_async: the upload overlaps the next query.  The engine keeps references to the host
        arrays until then (they must not be modified in between)."""
        defs = _f64(defs)
        if codes.dtype == np.uint8:
            cb = 1
        else:
            codes = np.ascontiguousarray(codes, dtype=np.int32)
            cb = 4
        codes = np.ascontiguousarray(codes)
        weights = None if weights is None else _f64(weights)
        self._pending_host = (codes, weights)
        self.S = codes.shape[0]
        self._ck(self._lib.plf_set_data_async(self._h, self.S, defs.shape[0], _ptr(defs), _ptr(codes), cb, _ptr(weights)))

    def set_data_async_ptr(self, defs, codes_ptr, S, weights_ptr=None, code_bytes=1):
        defs = _f64(defs)
        self.S = S
        self._ck(self._lib.plf_set_data_async(self._h, S, defs.shape[0], _ptr(defs), ctypes.c_void_p(codes_ptr), code_bytes,
                                              ctypes.c_void_p(weights_ptr) if weights_ptr else None))

    def set_site_weights(self, w):
        self._ck(self._lib.plf_set_site_weights(self._h, _ptr(_f64(w))))

    def ll(self, per_site=True):
        site = np.empty(self.S) if per_site else None
        tot = np.zeros(1)
        self._ck(self._lib.plf_ll(self._h, _ptr(site), _ptr(tot)))
        return site, float(tot[0])

    def deriv(self, edge_mask=None, per_site=True, per_site_ll=False):
        m = None if edge_mask is None else np.ascontiguousarray(edge_mask, dtype=np.uint8)
        sd = np.empty((self.S, self.E)) if per_site else None
        sl = np.empty(self.S) if per_site_ll else None
        sll = np.zeros(1)
        sde = np.zeros(self.E)
        self._ck(self._lib.plf_deriv(self._h, _ptr(m), _ptr(sl), _ptr(sll), _ptr(sd), _ptr(sde)))
        return dict(site_ll=sl, sum_ll=float(sll[0]), site_deriv=sd, sum_deriv=sde)

    def marginal(self, per_site=True):
        sm = np.empty((self.S, self.N, self.n)) if per_site else None
        tot = np.zeros((self.N, self.n))
        self._ck(self._lib.plf_marginal(self._h, _ptr(sm), _ptr(tot)))
        return sm, tot

    def edge_expect(self, kind, l_hi, l_lo=None, edge_mask=None, per_site=True):
        m = None if edge_mask is None else np.ascontiguousarray(edge_mask, dtype=np.uint8)
        so = np.empty((self.S, self.E)) if per_site else None
        tot = np.zeros(self.E)
        self._ck(self._lib.plf_edge_expect(self._h, kind, _ptr(_f64(l_hi)), _ptr(_f64(l_lo)), _ptr(m), _ptr(so), _ptr(tot)))
        return so, tot

    def edge_expect_all(self):
        """Every Frechet direction of edge_expect in one pass, site-summed with the site weights (plf_edge_expect_all):
        sum_ll, dwell [E, n, n] and trans [E, n, n] with edge_expect(kind, L)[1][e] == (L * X_kind[e]).sum(), and
        q_grad = trans.sum(0), the gradient of sum_ll with respect to the entries of the scaled rate matrix (category
        rates, category priors and root prior held fixed)."""
        sll = np.zeros(1)
        dwell = np.zeros((self.E, self.n, self.n))
        trans = np.zeros((self.E, self.n, self.n))
        self._ck(self._lib.plf_edge_expect_all(self._h, _ptr(sll), _ptr(dwell), _ptr(trans)))
        return dict(sum_ll=float(sll[0]), dwell=dwell, trans=trans, q_grad=trans.sum(axis=0))

    def transition_matrices(self):
        out = np.empty((self.C, self.E, self.n, self.n))
        self._ck(self._lib.plf_get_transition_matrices(self._h, _ptr(out)))
        return out

    def derivative_matrices(self):
        out = np.empty((self.C, self.E, self.n, self.n))
        self._ck(self._lib.plf_get_derivative_matrices(self._h, _ptr(out)))
        return out

    def frechet_matrices(self, l_hi, l_lo=None):
        out = np.empty((self.C, self.E, self.n, self.n))
        self._ck(self._lib.plf_get_frechet_matrices(self._h, _ptr(_f64(l_hi)), _ptr(_f64(l_lo)), _ptr(out)))
        return out

    def ll_certified(self, delta_rate=4e-15, delta_q=2.0 ** -60):
        """Enclosures of the site log-likelihoods and of their weighted sum: (site_lo, site_hi, sum_lo, sum_hi)."""
        lo = np.zeros(self.S)
        hi = np.zeros(self.S)
        slo = np.zeros(1)
        shi = np.zeros(1)
        self._ck(self._lib.plf_ll_certified(self._h, delta_rate, delta_q, _ptr(lo), _ptr(hi), _ptr(slo), _ptr(shi)))
        return lo, hi, float(slo[0]), float(shi[0])

    def deriv_certified(self, edge_mask=None, per_site=True, delta_rate=4e-15, delta_q=2.0 ** -60):
        """Enclosures of the per-site derivatives [S, E] (csr order; None unless per_site) and of their weighted sums [E]:
        dict(site_lo, site_hi, sum_lo, sum_hi).  Unrequested edges are 0 in both bounds."""
        m = None if edge_mask is None else np.ascontiguousarray(edge_mask, dtype=np.uint8)
        lo = np.zeros((self.S, self.E)) if per_site else None
        hi = np.zeros((self.S, self.E)) if per_site else None
        slo = np.zeros(self.E)
        shi = np.zeros(self.E)
        self._ck(self._lib.plf_deriv_certified(self._h, delta_rate, delta_q, _ptr(m), _ptr(lo), _ptr(hi), _ptr(slo), _ptr(shi)))
        return dict(site_lo=lo, site_hi=hi, sum_lo=slo, sum_hi=shi)

    def marginal_certified(self, per_site=True, delta_rate=4e-15, delta_q=2.0 ** -60):
        """Enclosures of the posterior marginals [S, N, n] (None unless per_site) and of their weighted sums [N, n]:
        dict(site_lo, site_hi, sum_lo, sum_hi)."""
        lo = np.zeros((self.S, self.N, self.n)) if per_site else None
        hi = np.zeros((self.S, self.N, self.n)) if per_site else None
        slo = np.zeros((self.N, self.n))
        shi = np.zeros((self.N, self.n))
        self._ck(self._lib.plf_marginal_certified(self._h, delta_rate, delta_q, _ptr(lo), _ptr(hi), _ptr(slo), _ptr(shi)))
        return dict(site_lo=lo, site_hi=hi, sum_lo=slo, sum_hi=shi)

    def edge_expect_certified(self, kind, L, edge_mask=None, per_site=True, L_lo=None, delta_rate=4e-15, delta_q=2.0 ** -60):
        """Enclosures of edge_expect(kind, L): per site [S, E] (csr order; None unless per_site) and the weighted sums [E],
        dict(site_lo, site_hi, sum_lo, sum_hi).  L may have entries of both signs; unrequested edges are 0 in both bounds."""
        m = None if edge_mask is None else np.ascontiguousarray(edge_mask, dtype=np.uint8)
        lo = np.zeros((self.S, self.E)) if per_site else None
        hi = np.zeros((self.S, self.E)) if per_site else None
        slo = np.zeros(self.E)
        shi = np.zeros(self.E)
        self._ck(self._lib.plf_edge_expect_certified(self._h, delta_rate, delta_q, kind, _ptr(_f64(L)), _ptr(_f64(L_lo)), _ptr(m),
                                                     _ptr(lo), _ptr(hi), _ptr(slo), _ptr(shi)))
        return dict(site_lo=lo, site_hi=hi, sum_lo=slo, sum_hi=shi)

    def hess(self):
        """sum_ll, gradient [E] and Hessian [E, E] of the weighted log likelihood w.r.t. the edge rates (csr order)."""
        ll = np.zeros(1)
        grad = np.zeros(self.E)
        H = np.zeros((self.E, self.E))
        self._ck(self._lib.plf_hess(self._h, _ptr(ll), _ptr(grad), _ptr(H)))
        return float(ll[0]), grad, H

    def compress_patterns(self, codes):
        """Merge identical columns: (codes of the patterns in order of first occurrence, counts, site -> pattern map)."""
        codes = np.ascontiguousarray(codes)
        if codes.dtype not in (np.uint8, np.int32):
            codes = codes.astype(np.int32)
        S, N = codes.shape
        npat = ctypes.c_int64(0)
        out = np.empty_like(codes)
        counts = np.zeros(S, dtype=np.int64)
        smap = np.zeros(S, dtype=np.int64)
        self._ck(self._lib.plf_compress_patterns(self._h, S, N, codes.ctypes.data_as(ctypes.c_void_p), codes.dtype.itemsize,
                                                 ctypes.byref(npat), out.ctypes.data_as(ctypes.c_void_p),
                                                 counts.ctypes.data_as(ctypes.c_void_p), smap.ctypes.data_as(ctypes.c_void_p)))
        P = int(npat.value)
        return out[:P].copy(), counts[:P].copy(), smap

    def last_timing(self):
        a = ctypes.c_float()
        b = ctypes.c_float()
        self._lib.plf_last_timing(self._h, ctypes.byref(a), ctypes.byref(b))
        return a.value, b.value

    def last_kernel_ms(self):
        a = ctypes.c_float()
        self._lib.plf_last_kernel_ms(self._h, ctypes.byref(a))
        return a.value

    def last_kernel_name(self):
        return (self._lib.plf_last_kernel_name(self._h) or b"").decode()

    def comm_pause(self, paused=True):
        self._ck(self._lib.plf_comm_pause(self._h, 1 if paused else 0))

    def launch_count(self, reset=False):
        return int(self._lib.plf_launch_count(self._h, 1 if reset else 0))

    def stream(self):
        return self._lib.plf_stream(self._h)

    def synchronize(self):
        self._ck(self._lib.plf_synchronize(self._h))

    def comm_init(self, nranks, rank, uid):
        self._ck(self._lib.plf_comm_init(self._h, nranks, rank, uid))


def comm_unique_id():
    lib = _lib.load()
    buf = ctypes.create_string_buffer(128)
    if lib.plf_comm_unique_id(buf) != 0:
        raise EngineError("plf_comm_unique_id failed")
    return buf.raw
