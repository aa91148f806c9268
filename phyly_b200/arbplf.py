"""
Python mirror of the reference's `arbplf` extension module (src/arbplf.c:521-546):
eleven functions, each `str -> str` (JSON in, JSON out), raising
RuntimeError("arbplf likelihood error") on a non-zero retcode
(src/arbplf.c:238-241).  Every call goes straight into libarbplf_b200.so
(include/arbplf.h); nothing is computed in Python.

    import phyly_b200.arbplf as arbplf
    out = arbplf.arbplf_ll(json.dumps(doc))
"""
import ctypes

from . import _lib

_NAMES = ["ll", "deriv", "marginal", "dwell", "trans", "hess", "inv_hess", "newton_delta",
          "newton_update", "newton_refine", "em_update"]
_MESSAGES = {"ll": "arbplf likelihood error"}

_libc = ctypes.CDLL(None)
_libc.free.argtypes = [ctypes.c_void_p]
_libc.free.restype = None


def _bind(name):
    def f(s_in):
        if isinstance(s_in, str):
            s_in = s_in.encode("utf-8")
        elif not isinstance(s_in, (bytes, bytearray)):
            raise TypeError("%s() argument must be str" % ("arbplf_" + name))
        lib = _lib.load()
        fn = getattr(lib, "arbplf_" + name)
        fn.argtypes = [ctypes.c_char_p, ctypes.POINTER(ctypes.c_int)]
        fn.restype = ctypes.c_void_p
        rc = ctypes.c_int(0)
        p = fn(bytes(s_in), ctypes.byref(rc))
        try:
            if rc.value != 0 or not p:
                raise RuntimeError("arbplf %s error" % ("likelihood" if name == "ll" else name.replace("_", " ")))
            return ctypes.string_at(p).decode("utf-8")
        finally:
            if p:
                _libc.free(p)      # the string is malloc'd by the library, caller frees (runjson.c:64-65)
    f.__name__ = "arbplf_" + name
    f.__doc__ = "JSON string -> JSON string; see include/arbplf.h"
    return f


for _n in _NAMES:
    globals()["arbplf_" + _n] = _bind(_n)

arbplf_model_summary = _bind("model_summary")
# certified mode (not in the reference module, whose every output is certified): arbplf-ll answered with an enclosure
arbplf_ll_certified = _bind("ll_certified")
# and arbplf-deriv, whose derivative bounds certify their sign
arbplf_deriv_certified = _bind("deriv_certified")
# and arbplf-marginal, arbplf-dwell, arbplf-trans
arbplf_marginal_certified = _bind("marginal_certified")
arbplf_dwell_certified = _bind("dwell_certified")
arbplf_trans_certified = _bind("trans_certified")


def set_device(device):
    _lib.load().arbplf_set_device(int(device))


__all__ = ["arbplf_" + n for n in _NAMES] + ["arbplf_model_summary", "arbplf_ll_certified", "arbplf_deriv_certified",
                                            "arbplf_marginal_certified", "arbplf_dwell_certified", "arbplf_trans_certified",
                                            "set_device"]
