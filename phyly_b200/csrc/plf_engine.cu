/*
 * plf_engine.cu -- implementation of the device seam declared in include/plf.h.
 *
 * Host side: buffer management, compilation of the tree into the fused-kernel
 * program, kernel launches on one CUDA stream, second-stage reductions and the
 * optional in-stream ncclAllReduce.  There is deliberately no CPU
 * implementation of any query in this file: without a CUDA device plf_create
 * fails and every entry point returns an error.
 */
#include <cuda_runtime.h>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <string>
#include <mutex>
#include <type_traits>
#include <vector>
#include <algorithm>
#include <dlfcn.h>

#include "../../include/plf.h"
#include "dd.h"
#include "expm.cuh"
#include "generic.cuh"
#include "fused4_args.h"
#include "tile.cuh"
#include "dmma.h"
#include "compress.cuh"
#include "certified.cuh"
#include <cfenv>

/* ------------------------------------------------------------------ */
/* small utilities                                                     */
/* ------------------------------------------------------------------ */

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes)
    {
        if (bytes <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        if (cudaMalloc(&p, want) != cudaSuccess) {
            if (cudaMalloc(&p, bytes) != cudaSuccess) { p = nullptr; return -1; }
            want = bytes;
        }
        cap = want;
        /* debugging aid: fresh device memory is usually zero, which hides reads of cells nobody wrote */
        static const bool poison = getenv("PLF_POISON") != nullptr;
        if (poison) { cudaMemset(p, 0xFF, want); cudaDeviceSynchronize(); }   /* also against non-blocking streams */
        return 0;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    ~DevBuf() { release(); }          /* plf_destroy deletes the engine with its device current */
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    template <typename T> T *as() const { return reinterpret_cast<T *>(p); }
};

/* NCCL through dlopen so that the library has no link-time dependency and
 * shares whatever libnccl.so.2 the process already loaded (e.g. torch's). */
typedef struct { char internal[128]; } plf_nccl_id;
typedef void *plf_nccl_comm;
struct NcclApi {
    void *lib = nullptr;
    int (*GetUniqueId)(plf_nccl_id *) = nullptr;
    int (*CommInitRank)(plf_nccl_comm *, int, plf_nccl_id, int) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, plf_nccl_comm, cudaStream_t) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, plf_nccl_comm, cudaStream_t) = nullptr;
    int (*CommDestroy)(plf_nccl_comm) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool load()
    {
        if (lib) return true;
        lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) return false;
        GetUniqueId = (int (*)(plf_nccl_id *))dlsym(lib, "ncclGetUniqueId");
        CommInitRank = (int (*)(plf_nccl_comm *, int, plf_nccl_id, int))dlsym(lib, "ncclCommInitRank");
        AllReduce = (int (*)(const void *, void *, size_t, int, int, plf_nccl_comm, cudaStream_t))dlsym(lib, "ncclAllReduce");
        AllGather = (int (*)(const void *, void *, size_t, int, plf_nccl_comm, cudaStream_t))dlsym(lib, "ncclAllGather");
        CommDestroy = (int (*)(plf_nccl_comm))dlsym(lib, "ncclCommDestroy");
        GetErrorString = (const char *(*)(int))dlsym(lib, "ncclGetErrorString");
        return GetUniqueId && CommInitRank && AllReduce && CommDestroy;
    }
};
static NcclApi g_nccl;

#define PLF_PEER_MAX 16
#define PLF_PEER_CAP 8192          /* doubles per (sender, parity) slot of an inbox */

/* a configuration of the fused kernel: block size, tables staged in shared memory (0: read through L1 / L2),
 * packed codes, matrices in constant memory, pending partials of the ll-only walk in a global stack */
struct F4Config { int bd, staged; bool pack, cm, gstack; };
/* one that exists for the model's category count and fits the program: its kernel, shared memory and CTAs per SM */
struct Cand : F4Config { f4_kernel_t k; size_t smem; int per_sm; };
/* tuning / candidate cache of the fused kernel for one query kind and category count */
struct F4Slot {
    std::string cand_key;             /* program version / C / K / E / forced index the candidates were scanned for */
    std::vector<Cand> cands;
    uint64_t tuned_version = ~(uint64_t)0;
    size_t tuned_pick = 0;
    int tuned_C = 0, tuned_K = 0;
};

struct plf_engine {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    int path = PLF_PATH_AUTO;
    int sm_count = 0;

    /* tree */
    int N = 0, E = 0, root = -1;
    std::vector<int> indptr, indices, preorder;
    DevBuf d_indptr, d_indices, d_preorder, d_node_has_data;
    bool tree_dirty = true;

    /* model */
    int n = 0, C = 0, root_mode = 0;
    std::vector<double> q_hi, q_lo, edge_rates, cat_rates, cat_prior, root_vec;
    DevBuf d_qhi, d_qlo, d_edge_rates, d_cat_rates, d_cat_prior, d_root_vec;
    DevBuf d_P, d_D, d_F, d_lhi, d_llo, d_expm_ws;
    bool model_dirty = true, P_valid = false, D_valid = false;

    /* data */
    int64_t S = 0;
    int K = 0, code_bytes = 1;
    DevBuf d_codes_in, d_codes, d_defs, d_def_const, d_def_ones, d_site_w;
    bool have_w = false;
    std::vector<unsigned char> def_const_h;

    /* data upload still in flight (plf_set_data_async): chunk k covers sites
     * [bounds[k], bounds[k+1]) and is complete on the device when chunk_ev[k] fires */
    cudaStream_t copy_stream = nullptr;
    std::vector<cudaEvent_t> chunk_ev;
    std::vector<int64_t> pend_bounds;
    bool pend_active = false;
    int pend_in_bytes = 1;
    unsigned char *flags_pinned = nullptr;

    /* fused program */
    std::vector<F4Op> ops;
    std::vector<F4Child> children;
    DevBuf d_ops, d_children, d_TP, d_TF, d_Pint, d_Fint, d_Ptip, d_block_marg, d_marg_site, d_edge_of_int, d_edge_of_tip, d_code_row_node, d_tip_of_edge, d_TPg, d_TFg, d_int_seq;
    std::vector<int> edge_of_int, edge_of_tip, code_row_node;
    std::vector<unsigned char> node_has_data_h;
    int stack_depth = 0, nslots = 0, max_degree = 0;
    bool TP_valid = false, program_dirty = true;
    bool dm_valid = false;       /* packed matrices / tip tables of the DMMA kernels (dmma.cuh) */
    DevBuf d_dmPf, d_dmTPf, d_dmTFf, d_dm_defsf, d_dm_rootf, d_dm_stack, d_dm_stackmeta, d_dm_slab, d_dm_slabmeta, d_dm_Of, d_dm_oidx, d_dm_otr, d_dm_ops, d_dm_ch;
    int dm_out_depth = 0;
    F4Prog prog_h;
    uint64_t program_version = 0;
    /* slot = 5 * kind (ll, edge forms, marginals, edge matrices) + categories of the launch */
    F4Slot f4_slot[20];
    DevBuf f4w_ll, f4w_edge, f4w_marg;      /* per-window per-site outputs when C > 4 (run_fused_windows) */
    DevBuf d_block_gmat, g_fe, d_gmat_W, d_gmat_out;   /* plf_edge_expect_all */

    /* scratch */
    DevBuf d_scratch, d_scratchS, d_block_ll, d_block_edge, d_edge_site, d_sum, d_site_ll, d_err, d_mask, d_retry;
    DevBuf g_Lg, g_Kg, g_Cg, g_Eg, g_Fg, g_FK, g_cat_lh, g_cat_k, g_site_m, g_site_k, g_edge_out, g_marg_out, g_tr;
    DevBuf h_Yg, h_dFg, h_dFk, h_part, h_gram, h_tree, h_out;
    DevBuf c_Plo, c_Phi, c_ws, c_cat_hi, c_site_lo, c_site_hi, c_small;
    DevBuf c_Dlo, c_Dhi, c_Flo, c_Fhi, c_FK, c_xlo, c_xhi, c_xk, c_mlo, c_mhi, c_mk, c_olo, c_ohi, c_part, c_sums, c_err;

    /* timing / accounting */
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    float ms_mat = 0.f, ms_sites = 0.f, ms_kernel = 0.f, ms_kernel_override = -1.f;
    bool kernel_timed = false;
    int64_t launches = 0;

    /* nccl */
    plf_nccl_comm comm = nullptr;
    int nranks = 1;
    bool comm_paused = false;
    std::string last_kernel;
    /* all-reduce of the (short) sum vectors over peer memory instead of NCCL (peer_allreduce_kernel) */
    int rank = 0;
    bool peer_ready = false;
    void *peer_local = nullptr;                 /* this rank's inbox + flags (cudaMalloc, exported through CUDA IPC) */
    void *peer_ptr[PLF_PEER_MAX] = {nullptr};   /* every rank's inbox as mapped here (own entry = peer_local) */
    DevBuf d_peer_ptrs;
    unsigned long long peer_seq = 0;
};

#define FAIL(e, ...) do { char _b[512]; snprintf(_b, sizeof(_b), __VA_ARGS__); (e)->err = _b; return -1; } while (0)
#define CK(e, call) do { cudaError_t _r = (call); if (_r != cudaSuccess) { \
        FAIL(e, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(_r)); } } while (0)
#define ENSURE(e, buf, bytes) do { if ((buf).ensure(bytes)) FAIL(e, "out of device memory allocating %zu bytes (%s)", (size_t)(bytes), #buf); } while (0)
#define KCHECK(e) do { (e)->launches++; CK(e, cudaGetLastError()); } while (0)

/* ------------------------------------------------------------------ */
/* small kernels                                                       */
/* ------------------------------------------------------------------ */

/* input of PLF_CODES_PACKED4: two codes per byte, node 2j in the low nibble of byte j, rows of (N + 1) / 2 bytes */
struct Packed4 { unsigned char b; };

/* codes_in[S][N] (4 bytes) -> codes[N][S] (1 or 4 bytes); also flags nodes that carry data */
template <typename TIn, typename TOut>
__global__ void transpose_codes_kernel(const TIn *in, TOut *out, int64_t s_begin, int64_t s_end, int64_t S, int N,
                                       const unsigned char *def_ones, int *node_flags, int K, int *bad_code)
{
    __shared__ int tile[32][33];
    const int64_t s0 = s_begin + (int64_t)blockIdx.x * 32;
    const int n0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        int64_t s = s0 + r;
        int nd = n0 + threadIdx.x;
        tile[r][threadIdx.x] = (s < s_end && nd < N) ? (int)in[(size_t)s * N + nd] : -1;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        int nd = n0 + r;
        int64_t s = s0 + threadIdx.x;
        int code = tile[threadIdx.x][r];
        bool has = false;
        if (nd < N && s < s_end && (unsigned)code >= (unsigned)K) { *bad_code = 1; code = 0; }   /* reported by the host */
        if (nd < N && s < s_end) {
            out[(size_t)nd * S + s] = (TOut)code;
            has = !def_ones[code];
        }
        unsigned any = __ballot_sync(0xffffffffu, has);
        if (any && threadIdx.x == 0 && nd < N) {
            if (node_flags[nd] == 0) atomicOr(&node_flags[nd], 1);
        }
    }
}

/* The same for 1-byte output codes (K <= 256) from 1-byte or packed input, the shapes an alignment has: a CTA brings the
 * rows of 128 sites (a contiguous run of the input) into shared memory and writes them out node by node, 32 consecutive
 * sites per store.  The 32 x 32 tiles of the kernel above spend their time starting CTAs of 1 KB each: 350 us for the
 * 127 MB of cfg2 against 60 us here, which the end-to-end step pays in full (the transposes sit between the chunk kernels). */
#define TR_SITES 128
#define TR_NODES 252
template <typename TIn>
__global__ void __launch_bounds__(256) transpose_codes_rows_kernel(const TIn *in, unsigned char *out, int64_t s_begin, int64_t s_end,
                                                                   int64_t S, int N, const unsigned char *def_ones, int *node_flags,
                                                                   int K, int *bad_code, int pad_words)
{
    extern __shared__ __align__(16) unsigned char tr_tile[];
    const int64_t s0 = s_begin + (int64_t)blockIdx.x * TR_SITES;
    const int n0 = blockIdx.y * TR_NODES, nt = min(TR_NODES, N - n0);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int pad = pad_words * 4;
    const int rows = (s_end - s0 < TR_SITES) ? (int)(s_end - s0) : TR_SITES;
    if (sizeof(TIn) == 1 && !std::is_same<TIn, Packed4>::value) {
        const unsigned char *src = reinterpret_cast<const unsigned char *>(in);
        for (int r = warp; r < rows; r += nw) {
            const unsigned char *row = src + (size_t)(s0 + r) * N + n0;
            for (int b = lane; b < nt; b += 32) tr_tile[r * pad + b] = row[b];
        }
    } else {
        const unsigned char *src = reinterpret_cast<const unsigned char *>(in);
        const int rb = (N + 1) >> 1, b0 = n0 >> 1, nb = (nt + 1) >> 1;          /* TR_NODES is even: tiles start on a byte */
        for (int r = warp; r < rows; r += nw) {
            const unsigned char *row = src + (size_t)(s0 + r) * rb + b0;
            for (int b = lane; b < nb; b += 32) {
                const unsigned char v = row[b];
                tr_tile[r * pad + 2 * b] = v & 15;
                if (2 * b + 1 < nt) tr_tile[r * pad + 2 * b + 1] = v >> 4;
            }
        }
    }
    __syncthreads();
    for (int nd = warp; nd < nt; nd += nw) {
        unsigned any = 0;
#pragma unroll
        for (int k = 0; k < TR_SITES / 32; k++) {
            const int r = lane + 32 * k;
            bool has = false;
            if (r < rows) {
                int code = tr_tile[r * pad + nd];
                if (code >= K) { *bad_code = 1; code = 0; }          /* reported by the host */
                out[(size_t)(n0 + nd) * S + s0 + r] = (unsigned char)code;
                has = !def_ones[code];
            }
            any |= __ballot_sync(0xffffffffu, has);
        }
        if (any && lane == 0 && node_flags[n0 + nd] == 0) atomicOr(&node_flags[n0 + nd], 1);
    }
}

/* Multi-GPU queries over an upload still in flight: one word, summed with the results by the same all-reduce, tells every
 * rank whether ANY rank has to repeat the query (its pattern of data-carrying nodes changed: +1) or met a character
 * code outside the definition table (+2^20), so that all ranks issue the same sequence of collectives. */
__global__ void retry_word_kernel(const int *flags, const unsigned char *old_flags, int N, const int *bad, double *out)
{
    __shared__ int any;
    if (threadIdx.x == 0) any = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < N; i += blockDim.x)
        if ((flags[i] != 0) != (old_flags[i] != 0)) any = 1;
    __syncthreads();
    if (threadIdx.x == 0) *out = (any ? 1.0 : 0.0) + (*bad ? 1048576.0 : 0.0);
}

__global__ void flags_to_bytes_kernel(const int *flags, unsigned char *out, int N)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) out[i] = flags[i] ? 1 : 0;
}

/* compact tip tables: out[c][te][k][i] = sum_j M[c][edge_of_tip[te]][i][j] def[k][j].
 * mode 0: stochastic matrix (constant rows map to the constant);
 * mode 1: zero-row-sum matrix (constant rows map to exact 0); mode 2: no shortcut. */
__global__ void tip_table_kernel(const double *M, const double *defs, const unsigned char *def_const,
                                 const int *edge_of_tip, int C, int E, int Et, int K, int n,
                                 int mode, double *out)
{
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t total = (size_t)C * Et * K * n;
    if (idx >= total) return;
    int i = idx % n; size_t r = idx / n;
    int k = r % K; r /= K;
    int te = r % Et; int c = r / Et;
    const double *row = M + (((size_t)c * E + edge_of_tip[te]) * n + i) * n;
    const double *d = defs + (size_t)k * n;
    double v;
    if (def_const[k] && mode == 0) v = d[0];
    else if (def_const[k] && mode == 1) v = 0.0;
    else {
        v = 0.0;
        for (int j = 0; j < n; j++) v = fma(row[j], d[j], v);
    }
    out[idx] = v;
}

/* weighted row sums: out[r] += sum_s w[s0+s] * val[r][s]  (one CTA per row, fixed order) */
__global__ void wsum_rows_kernel(const double *val, const double *w, int64_t w_off, int cols, double *out, int *err, int check)
{
    __shared__ double red[256];
    const int r = blockIdx.x;
    const double *row = val + (size_t)r * cols;
    double s = 0.0;
    for (int j = threadIdx.x; j < cols; j += blockDim.x) {
        double wj = w ? w[w_off + j] : 1.0;
        if (wj != 0.0) {
            double v = row[j];
            if (check && !isfinite(v)) atomicOr(err, 1);
            s = fma(wj, v, s);
        }
    }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = blockDim.x / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[r] += red[0];
}

/*
 * Sites of zero likelihood.  The reference's precision loop never terminates on them (arbplfll.c:168, README.md:22-24);
 * here they are an error whenever they carry weight in an aggregate, and their per-site rows become NaN so that the
 * caller sees them whichever output it asked for.  ll[cols] are the site log-likelihoods of the chunk, w the weights of
 * all sites (or NULL = 1), rowsA [RA][cols] / rowsB [RB][cols] per-site outputs of the chunk (or NULL).
 */
__global__ void zero_lik_rows_kernel(const double *ll, const double *w, int64_t w_off, int cols, int *err,
                                     double *rowsA, int RA, double *rowsB, int RB)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= cols) return;
    if (isfinite(ll[s])) return;
    if (!w || w[w_off + s] != 0.0) atomicOr(err, 1);
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    if (rowsA) for (int r = 0; r < RA; r++) rowsA[(size_t)r * cols + s] = nan;
    if (rowsB) for (int r = 0; r < RB; r++) rowsB[(size_t)r * cols + s] = nan;
}

/*
 * All-reduce (sum) of a short vector over NVLink peer memory, fused with nothing but itself: one CTA per GPU.
 * Every rank stores its vector into the inbox of every rank (slot [sender][parity of the sequence number]), publishes
 * the sequence number in that inbox's flag for the sender with a system-scope release, waits until the flags of all
 * senders in its own inbox carry the sequence number, and adds the nranks vectors in rank order -- so every rank gets
 * the same bits.  Two parities suffice: a rank can only be one collective ahead of the slowest one, because the next
 * collective needs that rank's flag.  A bounded spin turns a lost peer into an error flag instead of a hung GPU.
 * Inbox layout: double data[PLF_PEER_MAX][2][PLF_PEER_CAP]; unsigned long long flag[PLF_PEER_MAX][2].
 */
/* Second stage of every reduction over per-CTA partial sums: the rows are dealt to PLF_ROW_GROUPS interleaved groups, each
 * summed in order with compensation by one thread, and the group sums are added in group order -- the same decomposition
 * in sum_rows_kernel and in the fused stage of peer_allreduce_kernel, so that both give the same bits (bench.py's
 * allreduce_check relies on it), and 8 times shorter than one thread walking all the rows. */
#define PLF_ROW_GROUPS 8
__device__ __forceinline__ double rows_group_sum(const double *col, size_t stride, int rows, int g)
{
    double s = 0.0, comp = 0.0;
    for (int r = g; r < rows; r += PLF_ROW_GROUPS) {
        const double yv = col[(size_t)r * stride] - comp, tsum = s + yv;
        comp = (tsum - s) - yv;
        s = tsum;
    }
    return s;
}

__global__ void peer_allreduce_kernel(double *vec, int count, unsigned long long seq, int rank, int nranks,
                                      void *const *inbox_of, int *err,
                                      const double *part_ll, const double *part_edge, int rows, int E)
{
    /* fused with the second stage of the reduction: vec[0] = sum of the per-CTA log-likelihood sums, vec[1 + e] = sum of
     * the per-CTA sums of edge e (fixed order, compensated), when the partial sums are handed in instead of a finished vec */
    if (part_ll) {
        /* launched with 128 * PLF_ROW_GROUPS threads for this form: thread = (column within a run of 128, row group) */
        __shared__ double sm[PLF_ROW_GROUPS][128];
        const int x = threadIdx.x & 127, g = threadIdx.x >> 7;
        for (int jb = 0; jb < count; jb += 128) {
            const int j = jb + x;
            if (g < PLF_ROW_GROUPS)
                sm[g][x] = (j < count) ? rows_group_sum((j == 0) ? part_ll : part_edge + (j - 1), (j == 0) ? (size_t)1 : (size_t)E, rows, g) : 0.0;
            __syncthreads();
            if (g == 0 && j < count) {
                double s = sm[0][x];
#pragma unroll
                for (int w = 1; w < PLF_ROW_GROUPS; w++) s += sm[w][x];
                vec[j] = s;
            }
            __syncthreads();
        }
    }
    const int par = (int)(seq & 1);
    const size_t flag_off = sizeof(double) * (size_t)PLF_PEER_MAX * 2 * PLF_PEER_CAP;
    for (int p = 0; p < nranks; p++) {
        double *dst = reinterpret_cast<double *>(inbox_of[p]) + ((size_t)rank * 2 + par) * PLF_PEER_CAP;
        for (int i = threadIdx.x; i < count; i += blockDim.x) dst[i] = vec[i];
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x < nranks) {
        unsigned long long *flag = reinterpret_cast<unsigned long long *>(reinterpret_cast<char *>(inbox_of[threadIdx.x]) + flag_off) + rank * 2 + par;
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(flag), "l"(seq) : "memory");
    }
    __shared__ int ok;
    if (threadIdx.x == 0) ok = 1;
    __syncthreads();
    if (threadIdx.x < nranks) {
        const unsigned long long *flag = reinterpret_cast<const unsigned long long *>(reinterpret_cast<const char *>(inbox_of[rank]) + flag_off) + threadIdx.x * 2 + par;
        unsigned long long v = 0;
        long long spins = 0;
        do {
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flag) : "memory");
        } while (v != seq && ++spins < 4000000LL);          /* a few seconds */
        if (v != seq) ok = 0;
    }
    __syncthreads();
    if (!ok) { if (threadIdx.x == 0) atomicOr(err, 4); return; }
    const double *mine = reinterpret_cast<const double *>(inbox_of[rank]);
    for (int i = threadIdx.x; i < count; i += blockDim.x) {
        double acc = 0.0;
        for (int r = 0; r < nranks; r++) acc += mine[((size_t)r * 2 + par) * PLF_PEER_CAP + i];
        vec[i] = acc;
    }
}

/* y += alpha x */
__global__ void axpy_kernel(double *y, const double *x, double alpha, size_t count)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) y[i] = fma(alpha, x[i], y[i]);
}

/* in[R][Cc] -> out[Cc][R] */
__global__ void transpose_d_kernel(const double *in, double *out, int R, int Cc)
{
    __shared__ double tile[32][33];
    int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        int rr = r0 + r, cc = c0 + threadIdx.x;
        tile[r][threadIdx.x] = (rr < R && cc < Cc) ? in[(size_t)rr * Cc + cc] : 0.0;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        int cc = c0 + r, rr = r0 + threadIdx.x;
        if (cc < Cc && rr < R) out[(size_t)cc * R + rr] = tile[threadIdx.x][r];
    }
}

/* second stage: out[j] = sum over rows of part[row][j], fixed order (Kahan) */
__global__ void __launch_bounds__(256) sum_rows_kernel(const double *part, int rows, int cols, double *out)
{
    /* block = (32 columns, PLF_ROW_GROUPS interleaved groups of rows); see rows_group_sum */
    __shared__ double sm[PLF_ROW_GROUPS][33];
    const int j = blockIdx.x * 32 + threadIdx.x, g = threadIdx.y;
    sm[g][threadIdx.x] = (j < cols) ? rows_group_sum(part + j, (size_t)cols, rows, g) : 0.0;
    __syncthreads();
    if (g == 0 && j < cols) {
        double s = sm[0][threadIdx.x];
#pragma unroll
        for (int w = 1; w < PLF_ROW_GROUPS; w++) s += sm[w][threadIdx.x];
        out[j] = s;
    }
}

/* gather the matrices of internal-child edges: out[c][ie] = M[c][edge_of[ie]] (16 doubles each) */
__global__ void compact_matrices_kernel(const double *M, const int *edge_of, int C, int E, int Ei, double *out)
{
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    int total = C * Ei * 16;
    if (idx >= total) return;
    int k = idx & 15, r = idx >> 4;
    int ie = r % Ei, c = r / Ei;
    out[idx] = M[((size_t)c * E + edge_of[ie]) * 16 + k];
}

/* the tables of the fused 4-state kernel in one launch: tip tables and compact internal-edge matrices of P and,
 * when Fm is given, of the edge-form matrices (four launches of the two kernels above otherwise) */
__global__ void f4_tables_kernel(const double *P, const double *Fm, const double *defs, const unsigned char *def_const,
                                 const int *edge_of_tip, const int *edge_of_int, int C, int E, int Et, int Ei, int K, int f_mode,
                                 double *TP, double *Pint, double *TF, double *Fint)
{
    const size_t cntT = (size_t)C * Et * K * 4, cntP = (size_t)C * Ei * 16;
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t per = cntT + cntP;
    if (idx >= per * (Fm ? 2 : 1)) return;
    const bool second = idx >= per;
    if (second) idx -= per;
    const double *M = second ? Fm : P;
    const int mode = second ? f_mode : 0;
    if (idx < cntT) {
        const int i = (int)(idx % 4); size_t r = idx / 4;
        const int k = (int)(r % K); r /= K;
        const int te = (int)(r % Et), c = (int)(r / Et);
        const double *row = M + (((size_t)c * E + edge_of_tip[te]) * 4 + i) * 4;
        const double *d = defs + (size_t)k * 4;
        double v;
        if (def_const[k] && mode == 0) v = d[0];
        else if (def_const[k] && mode == 1) v = 0.0;
        else { v = 0.0; for (int j = 0; j < 4; j++) v = fma(row[j], d[j], v); }
        (second ? TF : TP)[idx] = v;
    } else {
        idx -= cntT;
        const int k = (int)(idx & 15); const size_t r = idx >> 4;
        const int ie = (int)(r % Ei), c = (int)(r / Ei);
        (second ? Fint : Pint)[idx] = M[((size_t)c * E + edge_of_int[ie]) * 16 + k];
    }
}

/* ------------------------------------------------------------------ */
/* lifecycle                                                           */
/* ------------------------------------------------------------------ */

extern "C" int plf_warmup(int device)
{
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return -1;
    if (cudaSetDevice(device) != cudaSuccess || cudaFree(nullptr) != cudaSuccess) { cudaGetLastError(); return -1; }
    return 0;
}

extern "C" int plf_create(plf_engine **out, int device)
{
    if (!out) return -1;
    *out = nullptr;
    int ndev = 0;
    cudaError_t r = cudaGetDeviceCount(&ndev);
    if (r != cudaSuccess || ndev == 0) {
        fprintf(stderr, "plf_create: no CUDA device available (%s); this engine has no CPU path\n",
                r == cudaSuccess ? "device count is 0" : cudaGetErrorString(r));
        return -1;
    }
    if (device < 0 || device >= ndev) {
        fprintf(stderr, "plf_create: invalid device %d (have %d)\n", device, ndev);
        return -1;
    }
    plf_engine *e = new plf_engine();
    e->device = device;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess) {
        fprintf(stderr, "plf_create: cannot initialise device %d: %s\n", device, cudaGetErrorString(cudaGetLastError()));
        delete e;
        return -1;
    }
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    e->sm_count = prop.multiProcessorCount;
    for (int i = 0; i < 5; i++) cudaEventCreate(&e->ev[i]);
    *out = e;
    return 0;
}

extern "C" void plf_destroy(plf_engine *e)
{
    if (!e) return;
    cudaSetDevice(e->device);
    cudaStreamSynchronize(e->stream);
    for (int p = 0; p < e->nranks && p < PLF_PEER_MAX; p++)
        if (e->peer_ptr[p] && e->peer_ptr[p] != e->peer_local) cudaIpcCloseMemHandle(e->peer_ptr[p]);
    if (e->peer_local) cudaFree(e->peer_local);
    if (e->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(e->comm);
    DevBuf *bufs[] = {&e->d_indptr, &e->d_indices, &e->d_preorder, &e->d_node_has_data, &e->d_qhi, &e->d_qlo,
                      &e->d_edge_rates, &e->d_cat_rates, &e->d_cat_prior, &e->d_root_vec, &e->d_P, &e->d_D, &e->d_F,
                      &e->d_lhi, &e->d_llo, &e->d_expm_ws, &e->d_codes_in, &e->d_codes, &e->d_defs, &e->d_def_const,
                      &e->d_def_ones, &e->d_site_w, &e->d_ops, &e->d_children, &e->d_TP, &e->d_TF, &e->d_Ptip, &e->d_block_marg, &e->d_marg_site, &e->d_scratch,
                      &e->d_scratchS, &e->d_block_ll, &e->d_block_edge, &e->d_edge_site, &e->d_sum, &e->d_site_ll,
                      &e->d_err, &e->d_mask, &e->g_Lg, &e->g_Kg, &e->g_Cg, &e->g_Eg, &e->g_Fg, &e->g_FK, &e->g_cat_lh,
                      &e->g_cat_k, &e->g_site_m, &e->g_site_k, &e->g_edge_out, &e->g_marg_out, &e->g_tr};
    for (DevBuf *b : bufs) b->release();
    for (int i = 0; i < 5; i++) if (e->ev[i]) cudaEventDestroy(e->ev[i]);
    if (e->copy_stream) { cudaStreamSynchronize(e->copy_stream); cudaStreamDestroy(e->copy_stream); }
    for (cudaEvent_t v : e->chunk_ev) cudaEventDestroy(v);
    if (e->flags_pinned) cudaFreeHost(e->flags_pinned);
    cudaStreamDestroy(e->stream);
    delete e;
}

extern "C" const char *plf_last_error(const plf_engine *e) { return e ? e->err.c_str() : "null engine"; }

extern "C" int plf_set_path(plf_engine *e, int path)
{
    if (!e) return -1;
    if (path < PLF_PATH_AUTO || path > PLF_PATH_FUSED4) FAIL(e, "plf_set_path: invalid path %d", path);
    e->path = path;
    return 0;
}

extern "C" void *plf_stream(plf_engine *e) { return e ? (void *)e->stream : nullptr; }

extern "C" int plf_synchronize(plf_engine *e)
{
    if (!e) return -1;
    CK(e, cudaSetDevice(e->device));
    CK(e, cudaStreamSynchronize(e->stream));
    if (e->copy_stream) CK(e, cudaStreamSynchronize(e->copy_stream));   /* host buffers of an async upload are free again */
    return 0;
}

extern "C" int plf_last_timing(plf_engine *e, float *ms_matrices, float *ms_sites)
{
    if (!e) return -1;
    if (ms_matrices) *ms_matrices = e->ms_mat;
    if (ms_sites) *ms_sites = e->ms_sites;
    return 0;
}

extern "C" int plf_last_kernel_ms(plf_engine *e, float *ms_kernel)
{
    if (!e || !ms_kernel) return -1;
    *ms_kernel = e->ms_kernel;
    return 0;
}

extern "C" const char *plf_last_kernel_name(const plf_engine *e) { return e ? e->last_kernel.c_str() : ""; }

extern "C" int64_t plf_launch_count(plf_engine *e, int reset)
{
    if (!e) return -1;
    int64_t v = e->launches;
    if (reset) e->launches = 0;
    return v;
}

/* ------------------------------------------------------------------ */
/* tree                                                                */
/* ------------------------------------------------------------------ */

static int build_program(plf_engine *e)
{
    const int N = e->N;
    std::vector<int> need(N, 0), slot(N, -1);
    std::vector<std::vector<int>> ichild(N);   /* internal children (csr edge idx) sorted for visiting */
    e->max_degree = 0;
    auto is_leaf = [&](int v) { return e->indptr[v] == e->indptr[v + 1]; };
    for (int u = N - 1; u >= 0; u--) {
        int a = e->preorder[u];
        int deg = e->indptr[a + 1] - e->indptr[a];
        e->max_degree = std::max(e->max_degree, deg);
        std::vector<int> &ic = ichild[a];
        for (int idx = e->indptr[a]; idx < e->indptr[a + 1]; idx++)
            if (!is_leaf(e->indices[idx])) ic.push_back(idx);
        std::stable_sort(ic.begin(), ic.end(), [&](int x, int y) { return need[e->indices[x]] > need[e->indices[y]]; });
        int nd = 0;
        for (size_t j = 0; j < ic.size(); j++) nd = std::max(nd, (int)j + need[e->indices[ic[j]]]);
        need[a] = nd;
    }
    /* iterative DFS emitting internal nodes in post-order */
    std::vector<int> order;
    {
        std::vector<std::pair<int, size_t>> st;
        st.push_back({e->root, 0});
        while (!st.empty()) {
            auto &top = st.back();
            int a = top.first;
            if (top.second < ichild[a].size()) {
                int b = e->indices[ichild[a][top.second]];
                top.second++;
                st.push_back({b, 0});
            } else {
                order.push_back(a);
                st.pop_back();
            }
        }
    }
    e->ops.clear(); e->children.clear();
    e->edge_of_int.clear(); e->edge_of_tip.clear(); e->code_row_node.clear();
    for (size_t o = 0; o < order.size(); o++) slot[order[o]] = (int)o;
    std::vector<int> code_row(N, -1);
    auto row_of = [&](int node) {
        if (code_row[node] < 0) { code_row[node] = (int)e->code_row_node.size(); e->code_row_node.push_back(node); }
        return code_row[node];
    };
    std::vector<int> stk;
    int cur = -1, maxdepth = 0;
    for (size_t o = 0; o < order.size(); o++) {
        int a = order[o];
        F4Op op;
        op.node = a; op.first_child = (int)e->children.size(); op.nchild = 0; op.slot = (int)o;
        op.code_row = (!e->node_has_data_h.empty() && e->node_has_data_h[a]) ? row_of(a) : -1;
        op.spill_before = 0;
        const std::vector<int> &ic = ichild[a];
        int cur_edge = -1;
        for (int idx : ic) if (e->indices[idx] == cur) cur_edge = idx;
        if (cur != -1 && cur_edge == -1) {
            op.spill_before = 1;
            stk.push_back(cur);
            maxdepth = std::max(maxdepth, (int)stk.size());
        }
        auto add_internal = [&](int idx, int b, int kind) {
            F4Child ch;
            memset(&ch, 0, sizeof(ch));
            ch.kind = kind; ch.slot = slot[b]; ch.mat = (int)e->edge_of_int.size(); ch.code_row = -1; ch.edge = idx; ch.node = b;
            e->edge_of_int.push_back(idx);
            e->children.push_back(ch); op.nchild++;
        };
        if (cur_edge != -1) add_internal(cur_edge, cur, F4_KIND_CUR);
        size_t nstack = ic.size() - (cur_edge != -1 ? 1 : 0);
        for (size_t j = 0; j < nstack; j++) {
            if (stk.empty()) { e->err = "internal error: fused program stack underflow"; return -1; }
            int b = stk.back(); stk.pop_back();
            int be = -1;
            for (int idx : ic) if (e->indices[idx] == b) be = idx;
            if (be == -1) { e->err = "internal error: fused program stack mismatch"; return -1; }
            add_internal(be, b, F4_KIND_STACK);
        }
        for (int idx = e->indptr[a]; idx < e->indptr[a + 1]; idx++) {
            int b = e->indices[idx];
            if (is_leaf(b)) {
                F4Child ch;
                memset(&ch, 0, sizeof(ch));
                ch.kind = F4_KIND_TIP; ch.slot = -1; ch.mat = (int)e->edge_of_tip.size(); ch.code_row = row_of(b); ch.edge = idx; ch.node = b;
                e->edge_of_tip.push_back(idx);
                e->children.push_back(ch); op.nchild++;
            }
        }
        e->ops.push_back(op);
        cur = a;
    }
    if (!stk.empty()) { e->err = "internal error: fused program leaves a non-empty stack"; return -1; }
    e->stack_depth = maxdepth;
    e->nslots = (int)order.size();
    return 0;
}

extern "C" int plf_set_tree(plf_engine *e, int node_count, const int *indptr, const int *indices, const int *preorder)
{
    if (!e) return -1;
    if (node_count < 2 || !indptr || !indices || !preorder) FAIL(e, "plf_set_tree: invalid arguments");
    const int N = node_count, E = N - 1;
    if (indptr[0] != 0 || indptr[N] != E) FAIL(e, "plf_set_tree: indptr does not describe %d edges", E);
    std::vector<int> indeg(N, 0), seen(N, 0), pos(N, -1);
    for (int i = 0; i < N; i++) if (indptr[i + 1] < indptr[i]) FAIL(e, "plf_set_tree: indptr is not monotone");
    for (int j = 0; j < E; j++) {
        if (indices[j] < 0 || indices[j] >= N) FAIL(e, "plf_set_tree: child index out of range");
        indeg[indices[j]]++;
    }
    for (int u = 0; u < N; u++) {
        int a = preorder[u];
        if (a < 0 || a >= N || seen[a]) FAIL(e, "plf_set_tree: preorder is not a permutation");
        seen[a] = 1; pos[a] = u;
    }
    if (indeg[preorder[0]] != 0) FAIL(e, "plf_set_tree: preorder[0] is not the root");
    for (int a = 0; a < N; a++) {
        if (a != preorder[0] && indeg[a] != 1) FAIL(e, "plf_set_tree: not a rooted tree");
        for (int j = indptr[a]; j < indptr[a + 1]; j++)
            if (pos[indices[j]] <= pos[a]) FAIL(e, "plf_set_tree: preorder visits a child before its parent");
    }
    e->N = N; e->E = E; e->root = preorder[0];
    e->indptr.assign(indptr, indptr + N + 1);
    e->indices.assign(indices, indices + E);
    e->preorder.assign(preorder, preorder + N);
    e->node_has_data_h.clear();
    e->program_dirty = true;
    e->max_degree = 0;
    for (int a = 0; a < N; a++) e->max_degree = std::max(e->max_degree, indptr[a + 1] - indptr[a]);
    CK(e, cudaSetDevice(e->device));
    ENSURE(e, e->d_indptr, sizeof(int) * (N + 1));
    ENSURE(e, e->d_indices, sizeof(int) * E);
    ENSURE(e, e->d_preorder, sizeof(int) * N);
    CK(e, cudaMemcpyAsync(e->d_indptr.p, indptr, sizeof(int) * (N + 1), cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaMemcpyAsync(e->d_indices.p, indices, sizeof(int) * E, cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaMemcpyAsync(e->d_preorder.p, preorder, sizeof(int) * N, cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    e->P_valid = e->D_valid = e->TP_valid = e->dm_valid = false;
    e->S = 0;   /* data must be (re)set after the tree */
    return 0;
}

/* ------------------------------------------------------------------ */
/* model                                                               */
/* ------------------------------------------------------------------ */

extern "C" int plf_set_model(plf_engine *e, int n, int C, const double *q_hi, const double *q_lo,
                             const double *edge_rates, const double *cat_rates, const double *cat_prior,
                             int root_mode, const double *root_vec)
{
    if (!e) return -1;
    if (e->N == 0) FAIL(e, "plf_set_model: set the tree first");
    if (n < 1 || n > 128 || C < 1 || !q_hi || !edge_rates || !cat_rates || !cat_prior)
        FAIL(e, "plf_set_model: invalid arguments (n=%d C=%d)", n, C);
    if (root_mode < PLF_ROOT_NONE || root_mode > PLF_ROOT_CUSTOM) FAIL(e, "plf_set_model: invalid root mode");
    if ((root_mode == PLF_ROOT_EQUILIBRIUM || root_mode == PLF_ROOT_CUSTOM) && !root_vec)
        FAIL(e, "plf_set_model: root_vec is required for this root mode");
    for (int i = 0; i < e->E; i++) if (!(edge_rates[i] >= 0.0) || !std::isfinite(edge_rates[i]))
        FAIL(e, "plf_set_model: edge rate %d is not a finite non-negative number", i);
    for (int i = 0; i < C; i++) if (!(cat_rates[i] >= 0.0) || !std::isfinite(cat_rates[i]) || !(cat_prior[i] >= 0.0))
        FAIL(e, "plf_set_model: category %d has an invalid rate or prior", i);
    if (n != e->n) e->S = 0;
    e->n = n; e->C = C; e->root_mode = root_mode;
    e->q_hi.assign(q_hi, q_hi + n * n);
    if (q_lo) e->q_lo.assign(q_lo, q_lo + n * n); else e->q_lo.assign(n * n, 0.0);
    e->edge_rates.assign(edge_rates, edge_rates + e->E);
    e->cat_rates.assign(cat_rates, cat_rates + C);
    e->cat_prior.assign(cat_prior, cat_prior + C);
    e->root_vec.assign(n, 1.0);
    if (root_vec) e->root_vec.assign(root_vec, root_vec + n);
    CK(e, cudaSetDevice(e->device));
    ENSURE(e, e->d_qhi, sizeof(double) * n * n);
    ENSURE(e, e->d_qlo, sizeof(double) * n * n);
    ENSURE(e, e->d_edge_rates, sizeof(double) * e->E);
    ENSURE(e, e->d_cat_rates, sizeof(double) * C);
    ENSURE(e, e->d_cat_prior, sizeof(double) * C);
    ENSURE(e, e->d_root_vec, sizeof(double) * n);
    CK(e, cudaMemcpyAsync(e->d_qhi.p, e->q_hi.data(), sizeof(double) * n * n, cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaMemcpyAsync(e->d_qlo.p, e->q_lo.data(), sizeof(double) * n * n, cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaMemcpyAsync(e->d_edge_rates.p, e->edge_rates.data(), sizeof(double) * e->E, cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaMemcpyAsync(e->d_cat_rates.p, e->cat_rates.data(), sizeof(double) * C, cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaMemcpyAsync(e->d_cat_prior.p, e->cat_prior.data(), sizeof(double) * C, cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaMemcpyAsync(e->d_root_vec.p, e->root_vec.data(), sizeof(double) * n, cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    e->P_valid = e->D_valid = e->TP_valid = e->dm_valid = false;
    return 0;
}

extern "C" int plf_set_edge_rates(plf_engine *e, const double *edge_rates)
{
    if (!e) return -1;
    if (e->n == 0) FAIL(e, "plf_set_edge_rates: set the model first");
    for (int i = 0; i < e->E; i++) if (!(edge_rates[i] >= 0.0) || !std::isfinite(edge_rates[i]))
        FAIL(e, "plf_set_edge_rates: edge rate %d is not a finite non-negative number", i);
    e->edge_rates.assign(edge_rates, edge_rates + e->E);
    CK(e, cudaSetDevice(e->device));
    /* no wait here: a copy from pageable memory has left the host buffer (for the driver's staging area) when the call
     * returns, and everything that reads d_edge_rates is launched on the same stream */
    CK(e, cudaMemcpyAsync(e->d_edge_rates.p, e->edge_rates.data(), sizeof(double) * e->E, cudaMemcpyHostToDevice, e->stream));
    e->P_valid = e->D_valid = e->TP_valid = e->dm_valid = false;
    return 0;
}

/* launch the expm kernel; which outputs are produced depends on the pointers */
static int run_expm(plf_engine *e, double *P, double *D, double *F, int f_scale_mode, const unsigned char *d_mask,
                    const double *d_lhi, const double *d_llo, const double *d_lper = nullptr, int q_transpose = 0)
{
    ExpmArgs a;
    a.n = e->n; a.E = e->E; a.C = e->C;
    a.q_hi = e->d_qhi.as<double>(); a.q_lo = e->d_qlo.as<double>();
    a.l_hi = d_lhi; a.l_lo = d_llo;
    a.l_per = d_lper; a.q_transpose = q_transpose;
    a.edge_rate = e->d_edge_rates.as<double>(); a.cat_rate = e->d_cat_rates.as<double>();
    a.edge_mask = d_mask;
    a.P = P; a.D = D; a.F = F; a.f_scale_mode = f_scale_mode;
    const size_t nn = (size_t)e->n * e->n;
    if (e->n == 4 && !F && !getenv("PLF_NO_EXPM4")) {
        /* P (and D) of a 4-state model: half a warp per matrix, eight matrices per CTA */
        a.ws = nullptr;
        expm4_dd_kernel<<<(e->C * e->E + 7) / 8, 128, 0, e->stream>>>(a);
        KCHECK(e);
        return 0;
    }
    size_t smem = 0;
    if (e->n <= 16) { a.ws = nullptr; smem = 8 * nn * sizeof(dd_t); }
    else {
        ENSURE(e, e->d_expm_ws, (size_t)e->C * e->E * 8 * nn * sizeof(dd_t));
        a.ws = e->d_expm_ws.as<dd_t>();
    }
    int threads = (int)std::min<size_t>(256, ((nn + 31) / 32) * 32);
    dim3 grid(e->E, e->C);
    expm_dd_kernel<<<grid, threads, smem, e->stream>>>(a);
    KCHECK(e);
    return 0;
}

static int ensure_matrices(plf_engine *e, bool need_D)
{
    const size_t bytes = sizeof(double) * e->C * e->E * e->n * e->n;
    if (e->P_valid && (!need_D || e->D_valid)) return 0;
    ENSURE(e, e->d_P, bytes);
    if (need_D) ENSURE(e, e->d_D, bytes);
    if (run_expm(e, e->d_P.as<double>(), need_D ? e->d_D.as<double>() : nullptr, nullptr, 0, nullptr, nullptr, nullptr)) return -1;
    e->P_valid = true;
    if (need_D) e->D_valid = true;
    e->TP_valid = e->dm_valid = false;
    return 0;
}

static int upload_L(plf_engine *e, const double *l_hi, const double *l_lo)
{
    const size_t nn = (size_t)e->n * e->n;
    if (!l_hi) FAIL(e, "Frechet direction matrix is required");
    std::vector<double> zero(nn, 0.0);
    ENSURE(e, e->d_lhi, sizeof(double) * nn);
    ENSURE(e, e->d_llo, sizeof(double) * nn);
    CK(e, cudaMemcpyAsync(e->d_lhi.p, l_hi, sizeof(double) * nn, cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaMemcpyAsync(e->d_llo.p, l_lo ? l_lo : zero.data(), sizeof(double) * nn, cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    return 0;
}

/* ------------------------------------------------------------------ */
/* data                                                                */
/* ------------------------------------------------------------------ */

/* site-major -> node-major for sites [s0, s1) on the engine's stream; accumulates the "node carries data" flags */
static int launch_transpose(plf_engine *e, int64_t s0, int64_t s1, int in_bytes)
{
    const int N = e->N;
    const int64_t S = e->S;
    int *flags = e->d_err.as<int>() + 4;
    int *bad = e->d_err.as<int>() + 1;          /* set when a code is not a row of the definition table */
    dim3 blk(32, 8), grid((unsigned)((s1 - s0 + 31) / 32), (unsigned)((N + 31) / 32));
    if (in_bytes == PLF_CODES_PACKED4 || in_bytes == 1) {
        /* rows of 128 sites through shared memory; the row pitch is an odd number of words (conflict-free columns) */
        const int nt = std::min(N, TR_NODES);
        const int pad_words = ((nt + 3) / 4) | 1;
        dim3 g((unsigned)((s1 - s0 + TR_SITES - 1) / TR_SITES), (unsigned)((N + TR_NODES - 1) / TR_NODES));
        const size_t smem = (size_t)TR_SITES * pad_words * 4;
        if (in_bytes == 1)
            transpose_codes_rows_kernel<unsigned char><<<g, 256, smem, e->stream>>>(
                e->d_codes_in.as<unsigned char>(), e->d_codes.as<unsigned char>(), s0, s1, S, N, e->d_def_ones.as<unsigned char>(), flags, e->K, bad, pad_words);
        else
            transpose_codes_rows_kernel<Packed4><<<g, 256, smem, e->stream>>>(
                e->d_codes_in.as<Packed4>(), e->d_codes.as<unsigned char>(), s0, s1, S, N, e->d_def_ones.as<unsigned char>(), flags, e->K, bad, pad_words);
    } else if (e->code_bytes == 1)
        transpose_codes_kernel<int, unsigned char><<<grid, blk, 0, e->stream>>>(
            e->d_codes_in.as<int>(), e->d_codes.as<unsigned char>(), s0, s1, S, N, e->d_def_ones.as<unsigned char>(), flags, e->K, bad);
    else
        transpose_codes_kernel<int, int><<<grid, blk, 0, e->stream>>>(
            e->d_codes_in.as<int>(), e->d_codes.as<int>(), s0, s1, S, N, e->d_def_ones.as<unsigned char>(), flags, e->K, bad);
    KCHECK(e);
    return 0;
}

/* after every chunk has been transposed: bring the node flags to the host (asynchronously) */
static int launch_flags_readback(plf_engine *e)
{
    int *flags = e->d_err.as<int>() + 4;
    flags_to_bytes_kernel<<<(e->N + 127) / 128, 128, 0, e->stream>>>(flags, e->d_node_has_data.as<unsigned char>(), e->N);
    KCHECK(e);
    CK(e, cudaMemcpyAsync(e->flags_pinned, e->d_node_has_data.p, e->N, cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaMemcpyAsync(e->flags_pinned + e->N, e->d_err.as<int>() + 1, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    return 0;
}

/* after the readback has completed: did the transposition meet a code outside the definition table? */
static bool data_has_bad_code(const plf_engine *e)
{
    int bad = 0;
    memcpy(&bad, e->flags_pinned + e->N, sizeof(int));
    return bad != 0;
}

/* the stream has been synchronised: compare the flags with the ones the program was built for */
static bool adopt_flags(plf_engine *e)
{
    std::vector<unsigned char> flags_h(e->flags_pinned, e->flags_pinned + e->N);
    if (flags_h == e->node_has_data_h) return false;
    e->node_has_data_h = flags_h;
    e->program_dirty = true;
    return true;
}

/* finish an upload started by plf_set_data_async without overlapping it with compute */
static int resolve_pending(plf_engine *e)
{
    if (!e->pend_active) return 0;
    for (size_t k = 0; k + 1 < e->pend_bounds.size(); k++) {
        CK(e, cudaStreamWaitEvent(e->stream, e->chunk_ev[k], 0));
        if (launch_transpose(e, e->pend_bounds[k], e->pend_bounds[k + 1], e->pend_in_bytes)) return -1;
    }
    if (launch_flags_readback(e)) return -1;
    CK(e, cudaStreamSynchronize(e->stream));
    adopt_flags(e);
    e->pend_active = false;
    if (data_has_bad_code(e)) { e->S = 0; FAIL(e, "plf_set_data_async: a character code is not a row of the definition table"); }
    return 0;
}

static int set_data_common(plf_engine *e, int64_t S, int K, const double *defs, const void *codes, int code_bytes,
                           const double *w, bool async)
{
    if (!e) return -1;
    if (e->N == 0 || e->n == 0) FAIL(e, "plf_set_data: set the tree and the model first");
    if (S < 1 || K < 1 || !defs || !codes || (code_bytes != 1 && code_bytes != 4 && code_bytes != PLF_CODES_PACKED4))
        FAIL(e, "plf_set_data: invalid arguments");
    if (code_bytes == 1 && K > 256) FAIL(e, "plf_set_data: %d definitions do not fit 1-byte codes", K);
    if (code_bytes == PLF_CODES_PACKED4 && K > 16) FAIL(e, "plf_set_data: %d definitions do not fit 4-bit codes", K);
    const int n = e->n, N = e->N;
    CK(e, cudaSetDevice(e->device));
    std::vector<unsigned char> dconst(K), dones(K);
    for (int k = 0; k < K; k++) {
        bool c = true, o = true;
        for (int i = 0; i < n; i++) {
            double v = defs[(size_t)k * n + i];
            if (!(v >= 0.0) || !std::isfinite(v)) FAIL(e, "plf_set_data: definition %d has an invalid entry", k);
            if (v != defs[(size_t)k * n]) c = false;
            if (v != 1.0) o = false;
        }
        dconst[k] = c; dones[k] = o;
    }
    /* an earlier asynchronous upload may still be writing the buffers that are about to be reused */
    if (e->pend_active) { CK(e, cudaStreamSynchronize(e->copy_stream)); e->pend_active = false; }
    e->def_const_h = dconst;
    const int dev_bytes = (K <= 256) ? 1 : 4;
    ENSURE(e, e->d_defs, sizeof(double) * K * n);
    ENSURE(e, e->d_def_const, K);
    ENSURE(e, e->d_def_ones, K);
    const size_t row = code_bytes == PLF_CODES_PACKED4 ? (size_t)(N + 1) / 2 : (size_t)N * code_bytes;    /* bytes per site of the input */
    ENSURE(e, e->d_codes_in, (size_t)S * row);
    ENSURE(e, e->d_codes, (size_t)S * N * dev_bytes);
    ENSURE(e, e->d_node_has_data, N);
    ENSURE(e, e->d_err, sizeof(int) * (N + 4));
    if (!e->flags_pinned) CK(e, cudaMallocHost((void **)&e->flags_pinned, 1 << 16));
    if (N > (1 << 16) - 8) FAIL(e, "plf_set_data: more than 65528 nodes");
    e->S = S; e->K = K; e->code_bytes = dev_bytes;
    e->TP_valid = e->dm_valid = false;
    e->have_w = false;
    CK(e, cudaMemcpyAsync(e->d_defs.p, defs, sizeof(double) * K * n, cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaMemcpyAsync(e->d_def_const.p, dconst.data(), K, cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaMemcpyAsync(e->d_def_ones.p, dones.data(), K, cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaMemsetAsync(e->d_err.p, 0, sizeof(int) * (N + 4), e->stream));
    if (w) ENSURE(e, e->d_site_w, sizeof(double) * S);
    if (!async) {
        CK(e, cudaMemcpyAsync(e->d_codes_in.p, codes, (size_t)S * row, cudaMemcpyHostToDevice, e->stream));
        if (w) { CK(e, cudaMemcpyAsync(e->d_site_w.p, w, sizeof(double) * S, cudaMemcpyHostToDevice, e->stream)); e->have_w = true; }
        if (launch_transpose(e, 0, S, code_bytes)) return -1;
        if (launch_flags_readback(e)) return -1;
        /* a host-side range check of the codes would cost a pass over S*N bytes; the
         * caller (the JSON front end) has already validated them (parsemodel.c:600-613). */
        CK(e, cudaStreamSynchronize(e->stream));   /* dconst / dones are locals; the flags are needed now */
        adopt_flags(e);
        if (data_has_bad_code(e)) { e->S = 0; FAIL(e, "plf_set_data: a character code is not a row of the definition table"); }
        return 0;
    }
    /* asynchronous: chunks of whole waves of the fused kernel (sm_count CTAs x 384 sites), copied on a second
     * stream; the queries wait chunk by chunk, so that the kernel runs while later chunks are still in flight */
    if (!e->copy_stream) CK(e, cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
    /* whole waves for both the 384- and the 512-thread kernels; the remainder rides with the last chunk so
     * that only one launch ends on a partial wave */
    /* Chunks are whole waves of 512-thread CTAs and double in size: the copy runs about twice as fast as the
     * kernel, so chunk k+1 (twice chunk k) lands just before kernel k ends; the remainder rides with the last
     * chunk so that only one launch ends on a partial wave. */
    const int64_t wave = (int64_t)e->sm_count * 512;
    e->pend_bounds.clear();
    e->pend_bounds.push_back(0);
    {
        int64_t s = 0, len = wave;
        while (S - s - len >= len && e->pend_bounds.size() < 8) { s += len; e->pend_bounds.push_back(s); len *= 2; }
    }
    e->pend_bounds.push_back(S);
    const size_t nch = e->pend_bounds.size() - 1;
    while (e->chunk_ev.size() < nch + 1) {
        cudaEvent_t v;
        CK(e, cudaEventCreateWithFlags(&v, cudaEventDisableTiming));
        e->chunk_ev.push_back(v);
    }
    /* the copy stream must not overtake earlier work on the main stream that still reads the buffers */
    CK(e, cudaEventRecord(e->chunk_ev[nch], e->stream));
    CK(e, cudaStreamWaitEvent(e->copy_stream, e->chunk_ev[nch], 0));
    for (size_t k = 0; k < nch; k++) {
        const int64_t s0 = e->pend_bounds[k], s1 = e->pend_bounds[k + 1];
        CK(e, cudaMemcpyAsync((char *)e->d_codes_in.p + (size_t)s0 * row, (const char *)codes + (size_t)s0 * row,
                              (size_t)(s1 - s0) * row, cudaMemcpyHostToDevice, e->copy_stream));
        if (w) CK(e, cudaMemcpyAsync(e->d_site_w.as<double>() + s0, w + s0, sizeof(double) * (s1 - s0),
                                     cudaMemcpyHostToDevice, e->copy_stream));
        CK(e, cudaEventRecord(e->chunk_ev[k], e->copy_stream));
    }
    if (w) e->have_w = true;
    e->pend_in_bytes = code_bytes;
    e->pend_active = true;
    CK(e, cudaStreamSynchronize(e->stream));       /* dconst / dones are locals */
    return 0;
}

extern "C" int plf_set_data(plf_engine *e, int64_t S, int K, const double *defs, const void *codes, int code_bytes)
{
    return set_data_common(e, S, K, defs, codes, code_bytes, nullptr, false);
}

extern "C" int plf_set_data_async(plf_engine *e, int64_t S, int K, const double *defs, const void *codes, int code_bytes,
                                  const double *site_weights)
{
    return set_data_common(e, S, K, defs, codes, code_bytes, site_weights, true);
}

extern "C" int plf_set_site_weights(plf_engine *e, const double *w)
{
    if (!e) return -1;
    if (e->S == 0) FAIL(e, "plf_set_site_weights: set the data first");
    CK(e, cudaSetDevice(e->device));
    /* an upload in flight may still be writing the weights it carried: let it finish first */
    if (e->pend_active && e->copy_stream) CK(e, cudaStreamSynchronize(e->copy_stream));
    if (!w) { e->have_w = false; return 0; }
    ENSURE(e, e->d_site_w, sizeof(double) * e->S);
    CK(e, cudaMemcpyAsync(e->d_site_w.p, w, sizeof(double) * e->S, cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));      /* the caller may reuse (pinned) w as soon as we return */
    e->have_w = true;
    return 0;
}

/* ------------------------------------------------------------------ */
/* queries                                                             */
/* ------------------------------------------------------------------ */

struct Query {
    bool want_edge = false, want_marg = false;
    const double *Fm = nullptr;      /* device [C][E][n][n] */
    int f_zero_rowsum = 0;
    const unsigned char *edge_mask_h = nullptr;
    /* host outputs (any may be NULL) */
    double *site_ll = nullptr, *sum_ll = nullptr;
    double *site_edge = nullptr, *sum_edge = nullptr;   /* [S][E], [E] */
    double *site_marg = nullptr, *sum_marg = nullptr;   /* [S][N][n], [N][n] */
    double *sum_hess = nullptr;                         /* [E][E]: Hessian of the weighted log likelihood (generic path) */
    /* plf_edge_expect_all: [sum_ll | G] is reduced, then run_gmat_adjoint turns G into the dwell / trans matrices */
    bool want_gmat = false;
    double *dwell_out = nullptr, *trans_out = nullptr;  /* [E][n][n] */
};

static int ensure_program(plf_engine *e)
{
    if (!e->program_dirty) return 0;
    if (build_program(e)) return -1;
    ENSURE(e, e->d_ops, sizeof(F4Op) * e->ops.size());
    ENSURE(e, e->d_children, sizeof(F4Child) * e->children.size());
    ENSURE(e, e->d_edge_of_int, sizeof(int) * (e->edge_of_int.size() + 1));
    ENSURE(e, e->d_edge_of_tip, sizeof(int) * (e->edge_of_tip.size() + 1));
    ENSURE(e, e->d_code_row_node, sizeof(int) * (e->code_row_node.size() + 1));
    CK(e, cudaMemcpyAsync(e->d_ops.p, e->ops.data(), sizeof(F4Op) * e->ops.size(), cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaMemcpyAsync(e->d_children.p, e->children.data(), sizeof(F4Child) * e->children.size(), cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaMemcpyAsync(e->d_edge_of_int.p, e->edge_of_int.data(), sizeof(int) * e->edge_of_int.size(), cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaMemcpyAsync(e->d_edge_of_tip.p, e->edge_of_tip.data(), sizeof(int) * e->edge_of_tip.size(), cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaMemcpyAsync(e->d_code_row_node.p, e->code_row_node.data(), sizeof(int) * e->code_row_node.size(), cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    e->program_dirty = false;
    e->program_version++;
    e->TP_valid = e->dm_valid = false;
    return 0;
}

/* compact matrices of the internal-child edges and tip tables for the fused kernel */
static int ensure_tip_tables(plf_engine *e, const double *Fm, int f_mode, bool want_ptip = false)
{
    if (ensure_program(e)) return -1;
    const int Ei = (int)e->edge_of_int.size(), Et = (int)e->edge_of_tip.size();
    const size_t cntT = (size_t)e->C * Et * e->K * e->n, cntP = (size_t)e->C * Ei * 16;
    const int threads = 256;
    if (want_ptip) {
        /* marginal mode: the transition matrices of the tip edges themselves (a tip's posterior needs P^T fe) */
        const size_t cntPt = (size_t)e->C * Et * 16;
        ENSURE(e, e->d_Ptip, sizeof(double) * (cntPt + 1));
        if (cntPt) {
            compact_matrices_kernel<<<(unsigned)((cntPt + threads - 1) / threads), threads, 0, e->stream>>>(
                e->d_P.as<double>(), e->d_edge_of_tip.as<int>(), e->C, e->E, Et, e->d_Ptip.as<double>());
            KCHECK(e);
        }
    }
    if (!e->TP_valid && Fm && cntT && cntP && e->n == 4) {
        /* the usual case of an optimisation step (matrices changed, edge forms wanted): one launch for all four tables */
        ENSURE(e, e->d_TP, sizeof(double) * (cntT + 1));
        ENSURE(e, e->d_Pint, sizeof(double) * (cntP + 1));
        ENSURE(e, e->d_TF, sizeof(double) * (cntT + 1));
        ENSURE(e, e->d_Fint, sizeof(double) * (cntP + 1));
        const size_t total = 2 * (cntT + cntP);
        f4_tables_kernel<<<(unsigned)((total + threads - 1) / threads), threads, 0, e->stream>>>(
            e->d_P.as<double>(), Fm, e->d_defs.as<double>(), e->d_def_const.as<unsigned char>(), e->d_edge_of_tip.as<int>(),
            e->d_edge_of_int.as<int>(), e->C, e->E, Et, Ei, e->K, f_mode, e->d_TP.as<double>(), e->d_Pint.as<double>(),
            e->d_TF.as<double>(), e->d_Fint.as<double>());
        KCHECK(e);
        e->TP_valid = true;
        return 0;
    }
    if (!e->TP_valid) {
        ENSURE(e, e->d_TP, sizeof(double) * (cntT + 1));
        ENSURE(e, e->d_Pint, sizeof(double) * (cntP + 1));
        if (cntT) {
            tip_table_kernel<<<(unsigned)((cntT + threads - 1) / threads), threads, 0, e->stream>>>(
                e->d_P.as<double>(), e->d_defs.as<double>(), e->d_def_const.as<unsigned char>(),
                e->d_edge_of_tip.as<int>(), e->C, e->E, Et, e->K, e->n, 0, e->d_TP.as<double>());
            KCHECK(e);
        }
        if (cntP) {
            compact_matrices_kernel<<<(unsigned)((cntP + threads - 1) / threads), threads, 0, e->stream>>>(
                e->d_P.as<double>(), e->d_edge_of_int.as<int>(), e->C, e->E, Ei, e->d_Pint.as<double>());
            KCHECK(e);
        }
        e->TP_valid = true;
    }
    if (Fm) {
        ENSURE(e, e->d_TF, sizeof(double) * (cntT + 1));
        ENSURE(e, e->d_Fint, sizeof(double) * (cntP + 1));
        if (cntT) {
            tip_table_kernel<<<(unsigned)((cntT + threads - 1) / threads), threads, 0, e->stream>>>(
                Fm, e->d_defs.as<double>(), e->d_def_const.as<unsigned char>(),
                e->d_edge_of_tip.as<int>(), e->C, e->E, Et, e->K, e->n, f_mode, e->d_TF.as<double>());
            KCHECK(e);
        }
        if (cntP) {
            compact_matrices_kernel<<<(unsigned)((cntP + threads - 1) / threads), threads, 0, e->stream>>>(
                Fm, e->d_edge_of_int.as<int>(), e->C, e->E, Ei, e->d_Fint.as<double>());
            KCHECK(e);
        }
    }
    return 0;
}

static bool peer_path(const plf_engine *e, size_t count)
{
    return e->comm && !e->comm_paused && e->peer_ready && count <= PLF_PEER_CAP && !getenv("PLF_NO_PEER_ALLREDUCE");
}

static int finish_sums(plf_engine *e, double *d_sum, size_t count)
{
    if (peer_path(e, count)) {
        ENSURE(e, e->d_err, sizeof(int) * (e->N + 4));
        e->peer_seq++;
        peer_allreduce_kernel<<<1, 256, 0, e->stream>>>(d_sum, (int)count, e->peer_seq, e->rank, e->nranks,
                                                        e->d_peer_ptrs.as<void *>(), e->d_err.as<int>(), nullptr, nullptr, 0, 0);
        KCHECK(e);
        return 0;
    }
    if (e->comm && !e->comm_paused) {
        int r = g_nccl.AllReduce(d_sum, d_sum, count, /*ncclDouble*/ 8, /*ncclSum*/ 0, e->comm, e->stream);
        if (r != 0) FAIL(e, "ncclAllReduce failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
    }
    return 0;
}

static int copy_site_matrix(plf_engine *e, const double *d_rows /*[R][cols]*/, int R, int64_t cols, double *host /*[cols][R]*/)
{
    /* transpose in column chunks to bound the staging buffer */
    const int64_t chunk = std::max<int64_t>(32, std::min<int64_t>(cols, (int64_t)(64u << 20) / std::max(1, R)));
    ENSURE(e, e->g_tr, sizeof(double) * (size_t)chunk * R * 2);
    double *src_c = e->g_tr.as<double>();
    double *dst_c = src_c + (size_t)chunk * R;
    for (int64_t c0 = 0; c0 < cols; c0 += chunk) {
        int cc = (int)std::min<int64_t>(chunk, cols - c0);
        /* gather the column block into a dense [R][cc] array */
        CK(e, cudaMemcpy2DAsync(src_c, sizeof(double) * cc, d_rows + c0, sizeof(double) * cols,
                                sizeof(double) * cc, R, cudaMemcpyDeviceToDevice, e->stream));
        dim3 blk(32, 8), grid((cc + 31) / 32, (R + 31) / 32);
        transpose_d_kernel<<<grid, blk, 0, e->stream>>>(src_c, dst_c, R, cc);
        KCHECK(e);
        CK(e, cudaMemcpyAsync(host + (size_t)c0 * R, dst_c, sizeof(double) * (size_t)cc * R, cudaMemcpyDeviceToHost, e->stream));
        CK(e, cudaStreamSynchronize(e->stream));
    }
    return 0;
}

/* the buffers every query path ends in: site log-likelihoods, the sum vector (sum_doubles of it) and the error word
 * (bit 0: a weighted site with zero likelihood, 1: Hessian infeasible, 2: peer all-reduce timed out), cleared */
static int prepare_sums(plf_engine *e, size_t sum_doubles)
{
    ENSURE(e, e->d_site_ll, sizeof(double) * e->S);
    ENSURE(e, e->d_sum, sizeof(double) * sum_doubles);
    ENSURE(e, e->d_err, sizeof(int) * (e->N + 4));
    CK(e, cudaMemsetAsync(e->d_err.p, 0, sizeof(int), e->stream));
    return 0;
}

/* the end of every query path: the first count doubles of d_sum, the error word, the site log-likelihoods and the
 * Hessian to the host */
static int read_back(plf_engine *e, const Query &q, const double *d_sum, size_t count, std::vector<double> &hs, int &herr)
{
    CK(e, cudaEventRecord(e->ev[2], e->stream));
    hs.assign(count, 0.0); herr = 0;
    CK(e, cudaMemcpyAsync(hs.data(), d_sum, sizeof(double) * count, cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaMemcpyAsync(&herr, e->d_err.p, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    if (q.site_ll) CK(e, cudaMemcpyAsync(q.site_ll, e->d_site_ll.p, sizeof(double) * e->S, cudaMemcpyDeviceToHost, e->stream));
    if (q.sum_hess) CK(e, cudaMemcpyAsync(q.sum_hess, e->h_out.p, sizeof(double) * (size_t)e->E * e->E, cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    return 0;
}

/* errors of the query, then the host sums from the read-back sum vector [ll | edge (E) | marginals (N n)] */
static int unpack_sums(plf_engine *e, const Query &q, const std::vector<double> &hs, int herr)
{
    const int E = e->E;
    if (herr & 4) FAIL(e, "all-reduce over peer memory timed out (a rank is missing)");
    if ((herr & 2) && q.sum_hess) FAIL(e, "infeasible: a rate category with a non-zero rate has zero likelihood at a weighted site");
    if ((herr & 1) && (q.sum_ll || q.sum_edge || q.sum_marg || q.want_gmat)) FAIL(e, "a site with non-zero weight has zero likelihood");
    if (q.sum_ll) *q.sum_ll = hs[0];
    if (q.sum_edge) memcpy(q.sum_edge, hs.data() + 1, sizeof(double) * E);
    if (q.sum_marg) memcpy(q.sum_marg, hs.data() + 1 + E, sizeof(double) * (size_t)e->N * e->n);
    if (q.sum_hess)
        for (int i = 0; i < E; i++) for (int j = 0; j < i; j++) q.sum_hess[(size_t)j * E + i] = q.sum_hess[(size_t)i * E + j];
    return 0;
}

/* the constant-memory matrices are one per device and context: queries of different engines (different
 * streams) that use them are ordered through this event */
static std::mutex g_cm_mutex;
static cudaEvent_t g_cm_done[64];

/* query kind of the fused path, the kernel's mode: 0 = ll, 1 = edge forms, 2 = marginals, 3 = edge matrices
 * (1 to 3 run an outside pass: slab, no stack) */
static int f4_kind(const Query &q) { return q.want_gmat ? 3 : (q.want_marg ? 2 : (q.want_edge ? 1 : 0)); }

/* mirrors the shared-memory carve-up at the top of fused4_kernel */
static size_t f4_smem_bytes(const plf_engine *e, int kind, int bd, int staged, bool pack = false, bool cm = false,
                            bool gstack = false)
{
    const int sdepth = gstack ? 0 : e->stack_depth;
    const int C = std::min(e->C, 4), Ei = cm ? 0 : (int)e->edge_of_int.size(), Et = (int)e->edge_of_tip.size();
    size_t off = 0;
    off = f4_align16(off + (cm ? 0 : sizeof(F4Op) * e->ops.size()));
    off = f4_align16(off + (cm ? 0 : sizeof(F4Child) * e->children.size()));
    off = f4_align16(off + sizeof(double) * 4 * C * bd);
    off = f4_align16(off + (kind == 1 ? sizeof(double) * (bd / 32) * e->E : 0));
    off = f4_align16(off + (kind ? 0 : sizeof(double) * 4 * C * bd * sdepth));
    off = f4_align16(off + (kind ? 0 : sizeof(int) * bd * sdepth));
    off = f4_align16(off + (pack ? (e->code_row_node.size() + 1) / 2 : e->code_row_node.size()) * bd);
    off = f4_align16(off + e->K);
    off = f4_align16(off + sizeof(double) * 4 * e->K);
    const size_t nP = (size_t)C * Ei * 16 * sizeof(double), nT = (size_t)C * Et * e->K * 4 * sizeof(double);
    const size_t nF = kind == 2 ? (size_t)C * Et * 16 * sizeof(double) : nP;
    if (staged) off += nP + nT + ((kind == 1 || kind == 2) ? nF : 0) + ((kind == 1 && staged == 2) ? nT : 0);
    return off + 16;
}

/* an outside pass is checked with the layout of the edge forms, the largest unstaged one */
static bool fused_fits(const plf_engine *e, bool outside)
{
    return f4_smem_bytes(e, outside ? 1 : 0, 128, 0) <= 227 * 1024;
}

/* dwell[e] = sum_c W[c][e], trans[e] = sum_c rate_c t_e W[c][e] (categories in order) */
__global__ void gmat_combine_kernel(const double *W, const double *cat_rate, const double *edge_rate, int C, int E, int nn,
                                    double *dwell, double *trans)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= E * nn) return;
    const double t = edge_rate[idx / nn];
    double d = 0.0, x = 0.0;
    for (int c = 0; c < C; c++) {
        const double w = W[(size_t)c * E * nn + idx];
        d += w;
        x = fma(cat_rate[c] * t, w, x);
    }
    dwell[idx] = d;
    trans[idx] = x;
}

/*
 * plf_edge_expect_all, after the all-reduce of G: the edge form is bilinear, fe^T F_A(L) L_b = <L, F_{A^T}(fe L_b^T)>
 * (the adjoint of the Frechet derivative of exp at A is the one at A^T), so W_{e,c} = F_{A_{e,c}^T}(G_{e,c}) (double-
 * double, one CTA per matrix) holds the values of every direction at once.  Every rank runs it on the same bits.
 */
static int run_gmat_adjoint(plf_engine *e, const double *d_G)
{
    const size_t nn = (size_t)e->n * e->n;
    ENSURE(e, e->d_gmat_W, sizeof(double) * (size_t)e->C * e->E * nn);
    ENSURE(e, e->d_gmat_out, sizeof(double) * 2 * (size_t)e->E * nn);
    if (run_expm(e, nullptr, nullptr, e->d_gmat_W.as<double>(), 0, nullptr, nullptr, nullptr, d_G, 1)) return -1;
    const int total = (int)(e->E * nn);
    double *out = e->d_gmat_out.as<double>();
    gmat_combine_kernel<<<(total + 255) / 256, 256, 0, e->stream>>>(e->d_gmat_W.as<double>(), e->d_cat_rates.as<double>(),
                                                                   e->d_edge_rates.as<double>(), e->C, e->E, (int)nn, out, out + total);
    KCHECK(e);
    return 0;
}

/* host copies of the matrices of run_gmat_adjoint (in stream: final after the query's synchronisation) */
static int copy_gmat_out(plf_engine *e, const Query &q)
{
    const size_t cnt = (size_t)e->E * e->n * e->n;
    if (q.dwell_out) CK(e, cudaMemcpyAsync(q.dwell_out, e->d_gmat_out.p, sizeof(double) * cnt, cudaMemcpyDeviceToHost, e->stream));
    if (q.trans_out) CK(e, cudaMemcpyAsync(q.trans_out, e->d_gmat_out.as<double>() + cnt, sizeof(double) * cnt, cudaMemcpyDeviceToHost, e->stream));
    return 0;
}

/* candidate configurations of the fused kernel per query kind, preferred first.  PLF_F4_CONFIG (edge forms),
 * PLF_F4_CONFIG_LL and PLF_F4_CONFIG_MARG (marginals, edge matrices) force one by its index here (tuning aid): an
 * entry keeps its place where it has no kernel (pack needs K <= 16, cm a small binary tree). */
static const std::vector<F4Config> f4_configs[3] = {
    /* log-likelihood only: no slab; the pending partials of the post-order walk either sit in shared
     * memory (which limits the CTA to 256 threads at depth 3) or in a small L2-resident global stack */
    {{512, 2, true, true, true}, {512, 2, true, false, true}, {512, 2, false, true, true}, {384, 2, true, false, true},
     {384, 2, true, false, false}, {384, 1, false, false, false}, {256, 2, false, false, false}, {256, 2, false, false, true},
     {512, 0, true, false, true}, {384, 0, true, false, true}, {384, 0, false, false, true}, {256, 0, false, false, true},
     {128, 0, false, false, true}, {128, 0, false, false, false}},
    /* edge forms; from index 7 on, for larger trees (the tables no longer fit shared memory): tables through L1 / L2,
     * CTAs stay large */
    {{512, 2, true, true}, {512, 2, false, true}, {384, 2, false, true}, {384, 2, true, false}, {384, 1, false, false},
     {512, 1, false, false}, {256, 2, false, false},
     {512, 0, true, false}, {384, 0, true, false}, {384, 0, false, false}, {256, 0, false, false}, {128, 0, false, false}},
    /* marginals and edge matrices (modes 2 and 3): the same configurations (mode 3 has the 256- and 128-thread ones) */
    {{384, 1, true, false}, {384, 1, false, false}, {256, 1, false, false},
     {384, 0, true, false}, {384, 0, false, false}, {256, 0, false, false}, {128, 0, false, false}},
};

/* sites of the tuning sample */
static int64_t f4_tune_sites(const plf_engine *e) { return (int64_t)e->sm_count * 512 * 2; }

/*
 * Which configuration a fused query of this kind runs: the slot with its viable candidates, the index of the one to
 * run or tune = true.  The candidates that fit (shared memory, occupancy) depend only on the program, the model's
 * shape and the query kind: scanned once and remembered -- the occupancy queries of a dozen instantiations cost more
 * host time per query than the matrix kernels take on the device.  The pick is the tuned one if this program has been
 * tuned, else the first.  Whether the constant-memory kernels beat the shared-memory ones depends on what the compiler
 * made of each instantiation (tools/check_cm_uniform.sh), so the first large query times the leading candidates on a
 * sample of the sites and keeps the fastest.
 */
static int f4_choose(plf_engine *e, int kind, F4Slot *&slot, size_t &pick, bool &tune)
{
    slot = &e->f4_slot[5 * kind + e->C];
    const char *force = getenv(kind >= 2 ? "PLF_F4_CONFIG_MARG" : (kind ? "PLF_F4_CONFIG" : "PLF_F4_CONFIG_LL"));
    const std::string cand_key = std::to_string(e->program_version) + "/" + std::to_string(e->C) + "/" + std::to_string(e->K) + "/" +
                                 std::to_string(e->E) + "/" + (force ? force : "");
    if (slot->cand_key != cand_key) {
        const bool can_pack = e->K <= 16;
        bool can_cm = (size_t)e->C * e->edge_of_int.size() * 16 <= F4_CM_MAXD && e->ops.size() <= F4_CM_MAXOPS &&
                      e->children.size() <= F4_CM_MAXCH && e->device < 64;
        for (const F4Op &op : e->ops) if (op.nchild != 2) can_cm = false;     /* CM kernels carry the two-children step only */
        const std::vector<F4Config> &cfgs = f4_configs[std::min(kind, 2)];
        std::vector<Cand> viable;
        size_t smem = 0;
        for (int i = 0; i < (int)cfgs.size(); i++) {
            const F4Config &f = cfgs[i];
            if ((force && atoi(force) != i) || (f.pack && !can_pack) || (f.cm && !can_cm)) continue;
            Cand c{f, f4_get_kernel(f.bd, f.staged, f.pack, f.cm, e->C, kind), 0, 0};
            if (!c.k) continue;
            c.smem = smem = f4_smem_bytes(e, kind, c.bd, c.staged, c.pack, c.cm, c.gstack);
            if (c.smem > 227 * 1024) continue;
            CK(e, cudaFuncSetAttribute(c.k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c.smem));
            CK(e, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c.per_sm, c.k, c.bd, c.smem));
            if (c.per_sm >= 1) viable.push_back(c);
        }
        if (viable.empty()) FAIL(e, "fused kernel: no configuration fits (C = %d, %zu bytes of shared memory)", e->C, smem);
        slot->cand_key = cand_key;
        slot->cands = std::move(viable);
    }
    const std::vector<Cand> &viable = slot->cands;
    const bool can_tune = viable.size() > 1 && e->S >= f4_tune_sites(e) / 2;
    pick = 0; tune = false;
    if (can_tune && slot->tuned_version == e->program_version && slot->tuned_C == e->C && slot->tuned_K == e->K &&
        slot->tuned_pick < viable.size())
        pick = slot->tuned_pick;
    else if (can_tune && !e->pend_active)
        tune = true;
    else        /* small problems, or untuned with the data still in flight: no constant-memory kernels */
        while (pick + 1 < viable.size() && viable[pick].cm) pick++;
    return 0;
}

/* A launch over a window of <= 4 rate categories [c0, c0 + e->C) of a model with more (run_fused_windows): per-site
 * outputs go to these device buffers. */
struct F4Window { int c0; double *site_ll, *site_edge, *site_marg; };

/* what the reduction of a fused query needs from its launches */
struct F4Launch { F4Args a; const Cand *use; int grid; size_t nchunk; bool pipelined; };

/* the arguments of a fused launch that do not depend on its configuration */
static void f4_fill_args(const plf_engine *e, const Query &q, int kind, const F4Window *win, F4Args &a)
{
    memset(&a, 0, sizeof(a));
    a.nops = (int)e->ops.size(); a.nchildren = (int)e->children.size();
    a.ops = e->d_ops.as<F4Op>(); a.children = e->d_children.as<F4Child>();
    a.E = e->E; a.K = e->K; a.S = e->S; a.N = e->N;
    a.Ei = (int)e->edge_of_int.size(); a.Et = (int)e->edge_of_tip.size();
    a.ncode_rows = (int)e->code_row_node.size();
    a.code_row_node = e->d_code_row_node.as<int>();
    a.codes = e->d_codes.as<unsigned char>();
    a.defs = e->d_defs.as<double>(); a.def_const = e->d_def_const.as<unsigned char>();
    a.Pint = e->d_Pint.as<double>(); a.TP = e->d_TP.as<double>();
    a.Fint = kind == 2 ? e->d_Ptip.as<double>() : (kind == 1 ? e->d_Fint.as<double>() : nullptr);
    a.TF = kind == 1 ? e->d_TF.as<double>() : nullptr;
    a.f_zero_rowsum = q.f_zero_rowsum;
    a.cat_prior = e->d_cat_prior.as<double>();
    a.root_mode = e->root_mode;
    for (int i = 0; i < 4; i++) a.root_vec[i] = e->root_vec[i];
    a.site_w = e->have_w ? e->d_site_w.as<double>() : nullptr;
    a.stack_depth = e->stack_depth; a.nslots = e->nslots;
    if (win) {
        /* the tables are laid out [category][...]: a window is a pointer offset */
        const size_t c0 = (size_t)win->c0;
        a.Pint += c0 * a.Ei * 16; a.TP += c0 * a.Et * a.K * 4;
        if (a.Fint) a.Fint += kind == 2 ? c0 * a.Et * 16 : c0 * a.Ei * 16;
        if (a.TF) a.TF += c0 * a.Et * a.K * 4;
        a.cat_prior += c0;
    }
}

/* grid of a fused launch over at most longest sites */
static int f4_grid(const plf_engine *e, const Cand &c, int64_t longest)
{
    return (int)std::min<int64_t>((longest + c.bd - 1) / c.bd, (int64_t)c.per_sm * e->sm_count);
}

/* times each leading candidate on the first sites (results are overwritten by the real run) and keeps the fastest */
static int f4_tune(plf_engine *e, F4Slot *slot, F4Args &a, int64_t longest, size_t &pick)
{
    const std::vector<Cand> &viable = slot->cands;
    float best = 0.f;
    const size_t ntry = std::min<size_t>(viable.size(), 5);
    a.s_begin = 0; a.s_end = std::min<int64_t>(e->S, f4_tune_sites(e));
    for (size_t i = 0; i < ntry; i++) {
        const Cand &c = viable[i];
        a.gstack = c.gstack ? 1 : 0; a.stack_depth = c.gstack ? 0 : e->stack_depth;
        /* candidates may share a kernel function with different amounts of dynamic shared memory */
        CK(e, cudaFuncSetAttribute(c.k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c.smem));
        float ms = 0.f;
        for (int rep = 0; rep < 4; rep++) {      /* the first launch pays for loading the code; then the best of three */
            float t = 0.f;
            CK(e, cudaEventRecord(e->ev[3], e->stream));
            c.k<<<f4_grid(e, c, longest), c.bd, c.smem, e->stream>>>(a, e->prog_h);
            KCHECK(e);
            CK(e, cudaEventRecord(e->ev[4], e->stream));
            CK(e, cudaEventSynchronize(e->ev[4]));
            CK(e, cudaEventElapsedTime(&t, e->ev[3], e->ev[4]));
            if (rep == 1 || (rep > 1 && t < ms)) ms = t;
        }
        if (i == 0 || ms < best) { best = ms; pick = i; }
    }
    slot->tuned_version = e->program_version; slot->tuned_C = e->C; slot->tuned_K = e->K;
    slot->tuned_pick = pick;
    return 0;
}

/*
 * The fused kernel over all sites for a query of this kind: arguments, the per-kind buffers, tuning when it is due,
 * then one launch per chunk of sites -- a single chunk normally, the upload's chunks while it is still in flight.
 * Nothing is reduced here.  prepare_sums has sized the site log-likelihoods and the error word.
 */
static int f4_launch(plf_engine *e, const Query &q, int kind, const F4Window *win, F4Launch &L)
{
    F4Slot *slot = nullptr; size_t pick = 0; bool tune = false;
    if (f4_choose(e, kind, slot, pick, tune)) return -1;
    const std::vector<Cand> &viable = slot->cands;
    F4Args &a = L.a;
    f4_fill_args(e, q, kind, win, a);
    L.pipelined = e->pend_active;
    std::vector<int64_t> bounds;
    if (L.pipelined) bounds = e->pend_bounds; else { bounds.push_back(0); bounds.push_back(e->S); }
    L.nchunk = bounds.size() - 1;
    int64_t longest = 0;
    for (size_t k = 0; k < L.nchunk; k++) longest = std::max(longest, bounds[k + 1] - bounds[k]);
    size_t Tmax = 0;
    int gmax = 0;
    bool any_cm = false, any_gstack = false;
    for (size_t i = 0; i < viable.size(); i++) {
        if (!tune && i != pick) continue;
        Tmax = std::max(Tmax, (size_t)f4_grid(e, viable[i], longest) * viable[i].bd);
        gmax = std::max(gmax, f4_grid(e, viable[i], longest));
        if (viable[i].cm) any_cm = true;
        if (viable[i].gstack) any_gstack = true;
    }

    ENSURE(e, e->d_block_ll, sizeof(double) * gmax * L.nchunk);
    const size_t ngm = kind == 3 ? (size_t)e->C * e->E * 16 : 0;     /* mode 3: a row [C][E][16] of G per warp */
    a.block_ll = e->d_block_ll.as<double>();
    a.error_flag = e->d_err.as<int>();
    /* the site log-likelihoods are always kept: the zero-likelihood check of every query kind reads them */
    a.site_ll = win ? win->site_ll : e->d_site_ll.as<double>();
    if (kind) {
        ENSURE(e, e->d_scratch, sizeof(double4) * (size_t)e->C * e->nslots * Tmax);
        ENSURE(e, e->d_scratchS, sizeof(unsigned int) * (size_t)e->nslots * Tmax);
        if (kind == 1) ENSURE(e, e->d_block_edge, sizeof(double) * (size_t)gmax * e->E * L.nchunk);
        a.scratch = e->d_scratch.as<double4>(); a.scratchS = e->d_scratchS.as<unsigned int>();
        a.block_edge = e->d_block_edge.as<double>();
        if (kind == 2 && win) {
            CK(e, cudaMemsetAsync(win->site_marg, 0, sizeof(double) * (size_t)e->N * 4 * e->S, e->stream));
            a.marg_site_out = win->site_marg;
        } else if (kind == 2 && q.site_marg) {
            ENSURE(e, e->d_marg_site, sizeof(double) * (size_t)e->N * 4 * e->S);
            CK(e, cudaMemsetAsync(e->d_marg_site.p, 0, sizeof(double) * (size_t)e->N * 4 * e->S, e->stream));
            a.marg_site_out = e->d_marg_site.as<double>();
        } else if (kind == 2) {
            /* one row of accumulators per warp of the grid; every launch of this query adds into them */
            const size_t rows = (size_t)gmax * 16;
            ENSURE(e, e->d_block_marg, sizeof(double) * rows * e->N * 4);
            CK(e, cudaMemsetAsync(e->d_block_marg.p, 0, sizeof(double) * rows * e->N * 4, e->stream));
            a.block_marg = e->d_block_marg.as<double>();
        } else if (kind == 3) {
            /* the same for the matrices G */
            ENSURE(e, e->d_block_gmat, sizeof(double) * (size_t)gmax * 16 * ngm);
            CK(e, cudaMemsetAsync(e->d_block_gmat.p, 0, sizeof(double) * (size_t)gmax * 16 * ngm, e->stream));
            a.block_gmat = e->d_block_gmat.as<double>();
        }
        a.edge_mask = q.edge_mask_h ? e->d_mask.as<unsigned char>() : nullptr;
        if (win && kind != 2) {
            CK(e, cudaMemsetAsync(win->site_edge, 0, sizeof(double) * (size_t)e->E * e->S, e->stream));
            a.edge_site_out = win->site_edge;
        } else if (q.site_edge) {
            ENSURE(e, e->d_edge_site, sizeof(double) * (size_t)e->E * e->S);
            CK(e, cudaMemsetAsync(e->d_edge_site.p, 0, sizeof(double) * (size_t)e->E * e->S, e->stream));
            a.edge_site_out = e->d_edge_site.as<double>();
        }
    }
    if (!kind && any_gstack && e->stack_depth > 0) {
        ENSURE(e, e->d_scratch, sizeof(double4) * (size_t)e->C * e->stack_depth * Tmax);
        ENSURE(e, e->d_scratchS, sizeof(unsigned int) * (size_t)e->stack_depth * Tmax);
        a.scratch = e->d_scratch.as<double4>(); a.scratchS = e->d_scratchS.as<unsigned int>();
    }
    std::unique_lock<std::mutex> cm_lock(g_cm_mutex, std::defer_lock);
    /* every way out of this function after the constant bank has been written records the "done" event before the
     * lock is released (declared after the lock: destroyed before it) */
    struct CmGuard {
        cudaEvent_t *ev = nullptr; cudaStream_t st = nullptr;
        ~CmGuard() { if (ev) cudaEventRecord(*ev, st); }
    } cm_guard;
    if (any_cm) {
        /* program as a kernel parameter, matrices into the constant bank (ordered against other engines) */
        memset(&e->prog_h, 0, sizeof(F4Prog));
        memcpy(e->prog_h.ops, e->ops.data(), sizeof(F4Op) * e->ops.size());
        memcpy(e->prog_h.ch, e->children.data(), sizeof(F4Child) * e->children.size());
        cm_lock.lock();
        if (!g_cm_done[e->device]) CK(e, cudaEventCreateWithFlags(&g_cm_done[e->device], cudaEventDisableTiming));
        CK(e, cudaStreamWaitEvent(e->stream, g_cm_done[e->device], 0));
        cm_guard.ev = &g_cm_done[e->device]; cm_guard.st = e->stream;
        const size_t nP = sizeof(double) * (size_t)e->C * e->edge_of_int.size() * 16;
        CK(e, f4_upload_const(a.Pint, kind ? a.Fint : nullptr, nP, e->stream));
    }
    if (tune) {
        if (f4_tune(e, slot, a, longest, pick)) return -1;
        CK(e, cudaMemsetAsync(e->d_err.p, 0, sizeof(int), e->stream));
        /* the marginal accumulators are added to by every launch: forget what the timing runs left there */
        if (kind == 2 && a.block_marg)
            CK(e, cudaMemsetAsync(e->d_block_marg.p, 0, sizeof(double) * (size_t)gmax * 16 * e->N * 4, e->stream));
        if (kind == 3) CK(e, cudaMemsetAsync(e->d_block_gmat.p, 0, sizeof(double) * (size_t)gmax * 16 * ngm, e->stream));
    }
    const Cand &use = viable[pick];
    const int grid = f4_grid(e, use, longest);
    {
        char nm[96];
        snprintf(nm, sizeof nm, "fused4_kernel<%d,%d,%d,%d,%d,%d>", e->C, kind, use.bd, use.staged, use.pack ? 1 : 0, use.cm ? 1 : 0);
        e->last_kernel = nm;
    }
    a.gstack = use.gstack ? 1 : 0; a.stack_depth = use.gstack ? 0 : e->stack_depth;
    CK(e, cudaFuncSetAttribute(use.k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)use.smem));
    CK(e, cudaEventRecord(e->ev[3], e->stream));
    for (size_t k = 0; k < L.nchunk; k++) {
        a.s_begin = bounds[k]; a.s_end = bounds[k + 1];
        a.block_ll = e->d_block_ll.as<double>() + k * (size_t)grid;
        if (kind == 1) a.block_edge = e->d_block_edge.as<double>() + k * (size_t)grid * e->E;
        if (L.pipelined) {
            /* this chunk's codes and weights have arrived; bring them into the node-major layout */
            CK(e, cudaStreamWaitEvent(e->stream, e->chunk_ev[k], 0));
            if (launch_transpose(e, a.s_begin, a.s_end, e->pend_in_bytes)) return -1;
        }
        use.k<<<grid, use.bd, use.smem, e->stream>>>(a, e->prog_h);
        KCHECK(e);
    }
    CK(e, cudaEventRecord(e->ev[4], e->stream));
    if (any_cm) {
        CK(e, cudaEventRecord(g_cm_done[e->device], e->stream));
        cm_guard.ev = nullptr;
        cm_lock.unlock();
    }
    e->kernel_timed = true;
    L.use = &use;
    L.grid = grid;
    return 0;
}

/* n = 4, up to 4 rate categories: the fused launches, then their rows reduced (and all-reduced) into the sums */
static int run_fused(plf_engine *e, Query &q)
{
    const int kind = f4_kind(q);
    const size_t ngm = kind == 3 ? (size_t)e->C * e->E * 16 : 0;     /* mode 3: G[C][E][16] follows sum_ll */
    if (prepare_sums(e, 2 + std::max((size_t)e->E + (size_t)e->N * e->n, ngm))) return -1;
    F4Launch L;
    if (f4_launch(e, q, kind, nullptr, L)) return -1;
    const F4Args &a = L.a;
    const int grid = L.grid;
    const bool pipelined = L.pipelined, shared_retry = pipelined && e->comm != nullptr;
    if (shared_retry) {
        ENSURE(e, e->d_retry, sizeof(double));
        retry_word_kernel<<<1, 256, 0, e->stream>>>(e->d_err.as<int>() + 4, e->d_node_has_data.as<unsigned char>(), e->N,
                                                    e->d_err.as<int>() + 1, e->d_retry.as<double>());
        KCHECK(e);
    }
    if (pipelined && launch_flags_readback(e)) return -1;
    if ((kind == 1 && q.site_edge) || (kind == 2 && q.site_marg)) {
        zero_lik_rows_kernel<<<(unsigned)((e->S + 255) / 256), 256, 0, e->stream>>>(
            a.site_ll, a.site_w, 0, (int)e->S, a.error_flag, kind == 1 ? a.edge_site_out : nullptr, e->E,
            kind == 2 ? a.marg_site_out : nullptr, e->N * 4);
        KCHECK(e);
    }
    const int rows = grid * (int)L.nchunk;
    double *block_ll = e->d_block_ll.as<double>(), *block_edge = e->d_block_edge.as<double>();
    double *dsum = e->d_sum.as<double>();
    /* ll / ll + edge sums with a communicator: second-stage reduction and all-reduce are one kernel over peer memory */
    const bool fuse_reduce = kind <= 1 && !q.site_edge && !pipelined && peer_path(e, 1 + (size_t)(kind ? e->E : 0));
    if (!fuse_reduce) {
        sum_rows_kernel<<<1, dim3(32, PLF_ROW_GROUPS), 0, e->stream>>>(block_ll, rows, 1, dsum);
        KCHECK(e);
    }
    size_t nsum = 1;
    if (kind == 2) {
        const int cols = e->N * 4;
        CK(e, cudaMemsetAsync(dsum + 1, 0, sizeof(double) * e->E, e->stream));
        if (q.site_marg) {
            if (q.sum_marg) {
                CK(e, cudaMemsetAsync(dsum + 1 + e->E, 0, sizeof(double) * cols, e->stream));
                wsum_rows_kernel<<<cols, 256, 0, e->stream>>>(a.marg_site_out, a.site_w, 0, (int)e->S, dsum + 1 + e->E, a.error_flag, 0);
                KCHECK(e);
            }
        } else {
            sum_rows_kernel<<<(cols + 31) / 32, dim3(32, PLF_ROW_GROUPS), 0, e->stream>>>(a.block_marg, grid * (L.use->bd / 32), cols, dsum + 1 + e->E);
            KCHECK(e);
        }
        nsum = 1 + e->E + cols;
    }
    if (kind == 3) {
        sum_rows_kernel<<<(unsigned)((ngm + 31) / 32), dim3(32, PLF_ROW_GROUPS), 0, e->stream>>>(a.block_gmat, grid * (L.use->bd / 32), (int)ngm, dsum + 1);
        KCHECK(e);
        nsum = 1 + ngm;
    }
    if (kind == 1 && !q.site_edge) {
        if (!fuse_reduce) {
            sum_rows_kernel<<<(e->E + 31) / 32, dim3(32, PLF_ROW_GROUPS), 0, e->stream>>>(block_edge, rows, e->E, dsum + 1);
            KCHECK(e);
        }
        nsum = 1 + e->E;
    }
    if (kind == 1 && q.site_edge && q.sum_edge) {
        /* per-site outputs requested together with sums: reduce the per-site rows with the weights */
        CK(e, cudaMemsetAsync(dsum + 1, 0, sizeof(double) * e->E, e->stream));
        wsum_rows_kernel<<<e->E, 256, 0, e->stream>>>(a.edge_site_out, a.site_w, 0, (int)e->S, dsum + 1, a.error_flag, 0);
        KCHECK(e);
        nsum = 1 + e->E;
    }
    if (shared_retry) CK(e, cudaMemcpyAsync(dsum + nsum, e->d_retry.p, sizeof(double), cudaMemcpyDeviceToDevice, e->stream));
    if (fuse_reduce) {
        e->peer_seq++;
        peer_allreduce_kernel<<<1, 128 * PLF_ROW_GROUPS, 0, e->stream>>>(dsum, (int)nsum, e->peer_seq, e->rank, e->nranks, e->d_peer_ptrs.as<void *>(),
                                                                         e->d_err.as<int>(), block_ll, kind ? block_edge : nullptr, rows, e->E);
        KCHECK(e);
    } else if (finish_sums(e, dsum, nsum + (shared_retry ? 1 : 0))) return -1;
    if (kind == 3 && (run_gmat_adjoint(e, dsum + 1) || copy_gmat_out(e, q))) return -1;
    std::vector<double> hs; int herr = 0;
    if (read_back(e, q, dsum, nsum + (shared_retry ? 1 : 0), hs, herr)) return -1;
    if (pipelined) {
        e->pend_active = false;
        if (data_has_bad_code(e)) { e->S = 0; FAIL(e, "plf_set_data_async: a character code is not a row of the definition table"); }
        if (shared_retry && hs[nsum] >= 1048576.0) { e->S = 0; FAIL(e, "plf_set_data_async: another rank met a character code that is not a row of the definition table"); }
        /* the program was compiled for the previous data's pattern of data-carrying nodes: redo if that changed here --
         * or, with a communicator, on any rank (the repeated query all-reduces again) */
        const bool changed = adopt_flags(e);
        if (changed || (shared_retry && hs[nsum] != 0.0)) return 1;
    }
    if (q.site_edge && copy_site_matrix(e, e->d_edge_site.as<double>(), e->E, e->S, q.site_edge)) return -1;
    if (unpack_sums(e, q, hs, herr)) return -1;
    if (kind == 2 && q.site_marg && copy_site_matrix(e, e->d_marg_site.as<double>(), e->N * 4, e->S, q.site_marg)) return -1;
    return 0;
}

/* combine the windows of a site: ll = log sum_w exp(ll_w); rows of window 0 <- sum_w exp(ll_w - ll) rows_w
 * (each window's per-site values are normalised by its own likelihood share) */
__global__ void f4_combine_windows_kernel(int nwin, int64_t S, double *w_ll /*[nwin][S]*/, double *site_ll /*[S]*/,
                                          double *rowsA /*[nwin][RA][S] or NULL*/, int RA, double *rowsB, int RB)
{
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    double mx = -INFINITY;
    for (int w = 0; w < nwin; w++) mx = fmax(mx, w_ll[(size_t)w * S + s]);
    double wt[16], tot = 0.0;
    for (int w = 0; w < nwin; w++) {
        const double l = w_ll[(size_t)w * S + s];
        wt[w] = (isfinite(mx) && isfinite(l)) ? exp(l - mx) : 0.0;
        tot += wt[w];
    }
    site_ll[s] = isfinite(mx) ? mx + log(tot) : -INFINITY;
    for (int w = 0; w < nwin; w++) wt[w] = tot > 0.0 ? wt[w] / tot : 0.0;
    if (rowsA) for (int r = 0; r < RA; r++) {
        double acc = 0.0;
        for (int w = 0; w < nwin; w++) if (wt[w] != 0.0) acc = fma(wt[w], rowsA[((size_t)w * RA + r) * S + s], acc);
        rowsA[(size_t)r * S + s] = acc;
    }
    if (rowsB) for (int r = 0; r < RB; r++) {
        double acc = 0.0;
        for (int w = 0; w < nwin; w++) if (wt[w] != 0.0) acc = fma(wt[w], rowsB[((size_t)w * RB + r) * S + s], acc);
        rowsB[(size_t)r * S + s] = acc;
    }
}

/*
 * n = 4 with more than 4 rate categories (GTR+Gamma4+I has 5, Gamma8 has 8): the fused kernel is instantiated for up to 4
 * categories in lock-step, so the categories are processed in windows of <= 4 -- each a launch of the tuned kernel with
 * per-site outputs -- and combined per site.  The site likelihood is a sum over categories, L = sum_w L_w, and every
 * per-site output a likelihood-weighted mean, x = sum_w x_w L_w / L, so the combination is exact up to rounding.
 */
static int run_fused_windows(plf_engine *e, Query &q)
{
    const int wsize = 4;
    const int Ctot = e->C, nwin = (Ctot + wsize - 1) / wsize, E = e->E, N = e->N;
    const int64_t S = e->S;
    const bool marg = q.want_marg, edge = q.want_edge && !marg;
    if (nwin > 16) FAIL(e, "more than 16 category windows");
    if (prepare_sums(e, 2 + E + (size_t)N * 4)) return -1;
    ENSURE(e, e->f4w_ll, sizeof(double) * (size_t)nwin * S);
    if (edge) ENSURE(e, e->f4w_edge, sizeof(double) * (size_t)nwin * E * S);
    if (marg) ENSURE(e, e->f4w_marg, sizeof(double) * (size_t)nwin * N * 4 * S);
    float ms_total = 0.f;
    for (int w = 0; w < nwin; w++) {
        F4Window win;
        win.c0 = wsize * w;
        win.site_ll = e->f4w_ll.as<double>() + (size_t)w * S;
        win.site_edge = edge ? e->f4w_edge.as<double>() + (size_t)w * E * S : nullptr;
        win.site_marg = marg ? e->f4w_marg.as<double>() + (size_t)w * N * 4 * S : nullptr;
        e->C = std::min(wsize, Ctot - wsize * w);
        F4Launch L;
        const int rc = f4_launch(e, q, f4_kind(q), &win, L);
        e->C = Ctot;
        if (rc) return rc;
        float t = 0.f;
        CK(e, cudaEventSynchronize(e->ev[4]));
        cudaEventElapsedTime(&t, e->ev[3], e->ev[4]);
        ms_total += t;
    }
    e->last_kernel += " (x" + std::to_string(nwin) + " category windows)";
    double *site_ll = e->d_site_ll.as<double>();
    f4_combine_windows_kernel<<<(unsigned)((S + 255) / 256), 256, 0, e->stream>>>(
        nwin, S, e->f4w_ll.as<double>(), site_ll, edge ? e->f4w_edge.as<double>() : nullptr, E,
        marg ? e->f4w_marg.as<double>() : nullptr, N * 4);
    KCHECK(e);
    const double *w = e->have_w ? e->d_site_w.as<double>() : nullptr;
    double *dsum = e->d_sum.as<double>();
    const size_t nsum = 1 + E + (size_t)N * 4;
    CK(e, cudaMemsetAsync(dsum, 0, sizeof(double) * nsum, e->stream));
    CK(e, cudaMemsetAsync(e->d_err.p, 0, sizeof(int), e->stream));
    zero_lik_rows_kernel<<<(unsigned)((S + 255) / 256), 256, 0, e->stream>>>(site_ll, w, 0, (int)S, e->d_err.as<int>(),
                                                                            edge ? e->f4w_edge.as<double>() : nullptr, E,
                                                                            marg ? e->f4w_marg.as<double>() : nullptr, N * 4);
    KCHECK(e);
    if (q.sum_ll) { wsum_rows_kernel<<<1, 256, 0, e->stream>>>(site_ll, w, 0, (int)S, dsum, e->d_err.as<int>(), 1); KCHECK(e); }
    if (edge && q.sum_edge) { wsum_rows_kernel<<<E, 256, 0, e->stream>>>(e->f4w_edge.as<double>(), w, 0, (int)S, dsum + 1, e->d_err.as<int>(), 0); KCHECK(e); }
    if (marg && q.sum_marg) { wsum_rows_kernel<<<N * 4, 256, 0, e->stream>>>(e->f4w_marg.as<double>(), w, 0, (int)S, dsum + 1 + E, e->d_err.as<int>(), 0); KCHECK(e); }
    if (finish_sums(e, dsum, nsum)) return -1;
    std::vector<double> hs; int herr = 0;
    if (read_back(e, q, dsum, nsum, hs, herr) || unpack_sums(e, q, hs, herr)) return -1;
    if (edge && q.site_edge && copy_site_matrix(e, e->f4w_edge.as<double>(), E, S, q.site_edge)) return -1;
    if (marg && q.site_marg && copy_site_matrix(e, e->f4w_marg.as<double>(), N * 4, S, q.site_marg)) return -1;
    e->ms_kernel_override = ms_total;
    return 0;
}

/* 16 < n <= 64 on the generic path: tip tables (when they are small) and the GEMM edge order of the tile kernels */
static int prepare_tile(plf_engine *e, const Query &q, GenericArgs &a)
{
    const int n = e->n, C = e->C, N = e->N, E = e->E;
    if (e->K <= 4096) {
        /* tip tables (P_e def_k) so that tip children need no GEMM */
        if (ensure_program(e)) return -1;
        const int Et = (int)e->edge_of_tip.size();
        std::vector<int> toe(E, -1);
        for (int te = 0; te < Et; te++) toe[e->edge_of_tip[te]] = te;
        ENSURE(e, e->d_tip_of_edge, sizeof(int) * E);
        CK(e, cudaMemcpyAsync(e->d_tip_of_edge.p, toe.data(), sizeof(int) * E, cudaMemcpyHostToDevice, e->stream));
        CK(e, cudaStreamSynchronize(e->stream));
        const size_t cnt = (size_t)C * Et * e->K * n;
        ENSURE(e, e->d_TPg, sizeof(double) * (cnt + 1));
        if (cnt) {
            tip_table_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, e->stream>>>(
                e->d_P.as<double>(), e->d_defs.as<double>(), e->d_def_const.as<unsigned char>(),
                e->d_edge_of_tip.as<int>(), C, E, Et, e->K, n, 0, e->d_TPg.as<double>());
            KCHECK(e);
        }
        a.TP = e->d_TPg.as<double>(); a.tip_of_edge = e->d_tip_of_edge.as<int>(); a.Et = Et;
        if (q.want_edge && a.Fm && cnt) {
            /* the same for the edge forms, so that tip edges need no GEMM in the outside pass either */
            ENSURE(e, e->d_TFg, sizeof(double) * (cnt + 1));
            tip_table_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, e->stream>>>(
                a.Fm, e->d_defs.as<double>(), e->d_def_const.as<unsigned char>(),
                e->d_edge_of_tip.as<int>(), C, E, Et, e->K, n, a.f_zero_rowsum ? 1 : 2, e->d_TFg.as<double>());
            KCHECK(e);
            a.TF = e->d_TFg.as<double>();
        }
    }
    /* GEMM edges in the order of the inside kernel's walk (reverse BFS, children in csr order) */
    std::vector<int> toe(E, -1);
    if (a.tip_of_edge) for (int te = 0; te < (int)e->edge_of_tip.size(); te++) toe[e->edge_of_tip[te]] = te;
    std::vector<int> seq, pos(N, 0);
    for (int u = 0; u < N; u++) pos[e->preorder[u]] = u;
    for (int u = N - 1; u >= 0; u--) {
        const int nd = e->preorder[u];
        for (int idx = e->indptr[nd]; idx < e->indptr[nd + 1]; idx++) if (toe[idx] < 0) seq.push_back(idx);
    }
    const size_t nseq = seq.size();
    for (size_t t = 0; t < nseq; t++) seq.push_back(pos[e->indices[seq[t]]]);    /* walk position of the child */
    ENSURE(e, e->d_int_seq, sizeof(int) * (seq.size() + 1));
    CK(e, cudaMemcpyAsync(e->d_int_seq.p, seq.data(), sizeof(int) * seq.size(), cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    a.int_seq = e->d_int_seq.as<int>(); a.n_int_seq = (int)nseq;
    if (a.tip_of_edge && e->code_bytes == 1 && (size_t)a.Et * TL_TS <= 32 * 1024) {
        a.tip_stage = 1;
        a.tip_edge_csr = e->d_edge_of_tip.as<int>();
    }
    return 0;
}

/* tree navigation arrays of the Hessian kernel, on the device */
static int upload_hess_tree(plf_engine *e, HessTree &ht)
{
    const int N = e->N, E = e->E;
    std::vector<int> nav((size_t)3 * E + (size_t)4 * N, 0);
    int *parent_node = nav.data(), *parent_edge = parent_node + E, *dfs_nodes = parent_edge + N, *dfs_pos = dfs_nodes + N,
        *sub_end = dfs_pos + N, *sub_max = sub_end + N, *erank = sub_max + E;
    for (int v = 0; v < N; v++) parent_edge[v] = -1;
    for (int v = 0; v < N; v++)
        for (int idx = e->indptr[v]; idx < e->indptr[v + 1]; idx++) { parent_node[idx] = v; parent_edge[e->indices[idx]] = idx; }
    /* depth-first pre-order (children in csr order), subtree ends */
    std::vector<int> st;
    int pos = 0;
    st.push_back(e->root);
    while (!st.empty()) {
        const int v = st.back(); st.pop_back();
        dfs_pos[v] = pos; dfs_nodes[pos++] = v;
        for (int idx = e->indptr[v + 1] - 1; idx >= e->indptr[v]; idx--) st.push_back(e->indices[idx]);
    }
    for (int p2 = N - 1; p2 >= 0; p2--) {
        const int v = dfs_nodes[p2];
        int end = p2 + 1;
        for (int idx = e->indptr[v]; idx < e->indptr[v + 1]; idx++) end = std::max(end, sub_end[e->indices[idx]]);
        sub_end[v] = end;
    }
    /* rank of an edge = BFS position of its child (csr indices follow the node labels, not the depth);
     * largest rank below (and including) every edge, children before parents */
    for (int u = 0; u < N; u++) { const int pe = parent_edge[e->preorder[u]]; if (pe >= 0) erank[pe] = u; }
    for (int u = N - 1; u >= 0; u--) {
        const int v = e->preorder[u], pe = parent_edge[v];
        if (pe < 0) continue;
        int mx = erank[pe];
        for (int i2 = e->indptr[v]; i2 < e->indptr[v + 1]; i2++) mx = std::max(mx, sub_max[i2]);
        sub_max[pe] = mx;
    }
    ENSURE(e, e->h_tree, sizeof(int) * nav.size());
    CK(e, cudaMemcpyAsync(e->h_tree.p, nav.data(), sizeof(int) * nav.size(), cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    const int *d = e->h_tree.as<int>();
    ht.parent_node = d; ht.parent_edge = d + E; ht.dfs_nodes = d + E + N; ht.dfs_pos = d + E + 2 * (size_t)N;
    ht.sub_end = d + E + 3 * (size_t)N; ht.sub_max = d + E + 4 * (size_t)N; ht.erank = d + 2 * (size_t)E + 4 * (size_t)N;
    return 0;
}

/* use_tile: 16 < n <= 64 (amino-acid, codon), inside pass on the FP64 tensor pipe (tile.cuh) */
static int run_generic(plf_engine *e, Query &q, bool use_tile)
{
    const int n = e->n, C = e->C, N = e->N, E = e->E;
    const bool gm = q.want_gmat;        /* plf_edge_expect_all: generic kernels only (generic_gmat_kernel) */
    const bool outside = q.want_edge || q.want_marg || gm;
    e->last_kernel = use_tile ? "tile_inside_kernel / tile_outside_kernel" : "generic_inside_kernel / generic_outside_kernel";
    const size_t ngm = gm ? (size_t)C * E * n * n : 0;     /* G[C][E][n][n] follows sum_ll */
    const size_t nsum_all = 1 + std::max((size_t)E + (size_t)N * n, ngm);
    /* chunk size from a memory budget */
    size_t per_site = (size_t)C * ((size_t)N * n * 8 + N * 5 + (size_t)E * n * 8 + 16) + 16;
    if (outside) per_site += (size_t)C * ((size_t)N * n * 8 + N * 4) + (size_t)E * 8 + (size_t)N * n * 8;
    if (q.sum_hess) per_site += (size_t)C * E * n * 8 + (size_t)N * n * 8 + (size_t)N * 4;
    if (gm) per_site += (size_t)C * E * n * 8;
    size_t free_b = 0, total_b = 0;
    CK(e, cudaMemGetInfo(&free_b, &total_b));
    size_t budget = std::min<size_t>((size_t)24 << 30, free_b / 2);
    int64_t Sc = std::max<int64_t>(PLF_TS, std::min<int64_t>(e->S, (int64_t)(budget / per_site)));
    Sc = std::min<int64_t>(Sc, 1 << 20);
    if (Sc < e->S) Sc = (Sc / PLF_TS) * PLF_TS;

    ENSURE(e, e->g_Lg, sizeof(double) * (size_t)C * N * n * Sc);
    ENSURE(e, e->g_Kg, sizeof(int) * (size_t)C * N * Sc);
    ENSURE(e, e->g_Cg, (size_t)C * N * Sc);
    ENSURE(e, e->g_Eg, sizeof(double) * (size_t)C * E * n * Sc);
    ENSURE(e, e->g_cat_lh, sizeof(double) * (size_t)C * Sc);
    ENSURE(e, e->g_cat_k, sizeof(int) * (size_t)C * Sc);
    ENSURE(e, e->g_site_m, sizeof(double) * Sc);
    ENSURE(e, e->g_site_k, sizeof(int) * Sc);
    if (prepare_sums(e, nsum_all)) return -1;
    if (gm) ENSURE(e, e->g_fe, sizeof(double) * (size_t)C * E * n * Sc);
    if (outside) {
        ENSURE(e, e->g_Fg, sizeof(double) * (size_t)C * N * n * Sc);
        ENSURE(e, e->g_FK, sizeof(int) * (size_t)C * N * Sc);
    }
    if (q.want_edge) ENSURE(e, e->g_edge_out, sizeof(double) * (size_t)E * Sc);
    if (q.want_marg) ENSURE(e, e->g_marg_out, sizeof(double) * (size_t)N * n * Sc);
    double *dsum = e->d_sum.as<double>();
    CK(e, cudaMemsetAsync(dsum, 0, sizeof(double) * nsum_all, e->stream));

    GenericArgs a;
    memset(&a, 0, sizeof(a));
    a.t.N = N; a.t.E = E; a.t.root = e->root;
    a.t.indptr = e->d_indptr.as<int>(); a.t.indices = e->d_indices.as<int>(); a.t.preorder = e->d_preorder.as<int>();
    a.t.node_has_data = e->d_node_has_data.as<unsigned char>();
    a.n = n; a.C = C; a.K = e->K; a.S = e->S;
    a.codes = e->d_codes.p; a.code_bytes = e->code_bytes;
    a.defs = e->d_defs.as<double>(); a.def_const = e->d_def_const.as<unsigned char>();
    a.P = e->d_P.as<double>(); a.Fm = q.Fm; a.f_zero_rowsum = q.f_zero_rowsum;
    a.edge_coef = nullptr;
    a.edge_mask = q.edge_mask_h ? e->d_mask.as<unsigned char>() : nullptr;
    a.cat_prior = e->d_cat_prior.as<double>();
    a.root_mode = e->root_mode; a.root_vec = e->d_root_vec.as<double>();
    a.Lg = e->g_Lg.as<double>(); a.Kg = e->g_Kg.as<int>(); a.Cg = e->g_Cg.as<unsigned char>();
    a.Eg = e->g_Eg.as<double>(); a.Fg = e->g_Fg.as<double>(); a.FK = e->g_FK.as<int>();
    a.cat_lh = e->g_cat_lh.as<double>(); a.cat_k = e->g_cat_k.as<int>();
    a.site_m = e->g_site_m.as<double>(); a.site_k = e->g_site_k.as<int>();
    a.site_ll = e->d_site_ll.as<double>();
    a.edge_out = q.want_edge ? e->g_edge_out.as<double>() : nullptr;
    a.marg_out = q.want_marg ? e->g_marg_out.as<double>() : nullptr;
    a.want_edge = q.want_edge; a.want_marg = q.want_marg;
    if (gm) { a.fe_out = e->g_fe.as<double>(); a.site_w = e->have_w ? e->d_site_w.as<double>() : nullptr; }

    const size_t smem_in = sizeof(double) * 2 * n * PLF_TS, smem_out = sizeof(double) * 3 * n * PLF_TS;
    if (smem_in > 48 * 1024) CK(e, cudaFuncSetAttribute(generic_inside_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_in));
    if (smem_out > 48 * 1024) CK(e, cudaFuncSetAttribute(generic_outside_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_out));
    if (smem_out > 227 * 1024) FAIL(e, "state count %d is too large for the generic kernels", n);
    const double *w = e->have_w ? e->d_site_w.as<double>() : nullptr;
    if (use_tile && prepare_tile(e, q, a)) return -1;
    /* padded state count of the tile kernels: 32 for amino-acid-sized models, 64 for codon-sized ones */
    const int tnp = n <= 32 ? 32 : 64, tnw = tnp / 8;
    const size_t smem_tile = sizeof(double) * (2 * tnp * TL_LS + tnw * TL_TS + TL_TS) + sizeof(int) * 2 * TL_TS +
                             (a.tip_stage ? (size_t)a.Et * TL_TS : 0) + 16;
    const size_t smem_tile_out = sizeof(double) * (tnp * TL_LS + tnw * TL_TS + 3 * TL_TS) + sizeof(int) * 6 * TL_TS;
    if (use_tile) {
        CK(e, cudaFuncSetAttribute(tile_inside_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tile));
        CK(e, cudaFuncSetAttribute(tile_outside_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tile_out));
        CK(e, cudaFuncSetAttribute(tile_inside_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tile));
        CK(e, cudaFuncSetAttribute(tile_outside_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tile_out));
    }

    /* second order (plf_hess): tree navigation arrays, per-CTA partial Hessians, the Gram matrix of the derivatives */
    HessTree ht;
    memset(&ht, 0, sizeof(ht));
    int hgrid = 0;
    const size_t smem_hess = sizeof(double) * ((size_t)3 * n * PLF_TS + E);
    if (q.sum_hess) {
        if (upload_hess_tree(e, ht)) return -1;
        hgrid = (int)std::min<int64_t>((Sc + PLF_TS - 1) / PLF_TS, (int64_t)e->sm_count * 4);
        while (hgrid > 1 && (size_t)hgrid * E * E * sizeof(double) > ((size_t)2 << 30)) hgrid /= 2;
        ENSURE(e, e->h_part, sizeof(double) * (size_t)hgrid * E * E + 8);
        ENSURE(e, e->h_gram, sizeof(double) * (size_t)E * E + 8);
        ENSURE(e, e->h_out, sizeof(double) * (size_t)E * E + 8);
        ENSURE(e, e->h_Yg, sizeof(double) * (size_t)C * E * n * Sc + 8);
        ENSURE(e, e->h_dFg, sizeof(double) * (size_t)N * n * Sc + 8);
        ENSURE(e, e->h_dFk, sizeof(int) * (size_t)N * Sc + 8);
        CK(e, cudaMemsetAsync(e->h_part.p, 0, sizeof(double) * (size_t)hgrid * E * E, e->stream));
        CK(e, cudaMemsetAsync(e->h_gram.p, 0, sizeof(double) * (size_t)E * E, e->stream));
        if (smem_hess > 227 * 1024) FAIL(e, "state count %d / edge count %d too large for the Hessian kernel", n, E);
        if (smem_hess > 48 * 1024) CK(e, cudaFuncSetAttribute(generic_hess_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_hess));
    }

    for (int64_t s0 = 0; s0 < e->S; s0 += Sc) {
        a.s0 = s0; a.Sc = (int)std::min<int64_t>(Sc, e->S - s0);
        const unsigned gx = (unsigned)((a.Sc + PLF_TS - 1) / PLF_TS);
        if (use_tile) {
            /* leaf vectors are only read when there are no tip tables, or by the marginal pass */
            generic_leaf_kernel<<<dim3((a.Sc + 255) / 256, C), 256, 0, e->stream>>>(
                a, (q.want_marg || !a.tip_of_edge || (q.want_edge && !a.TF)) ? 1 : 0);
            KCHECK(e);
            if (tnp == 32) tile_inside_kernel<32><<<dim3((a.Sc + TL_TS - 1) / TL_TS, C), 128, smem_tile, e->stream>>>(a, outside ? 1 : 0);
            else tile_inside_kernel<64><<<dim3((a.Sc + TL_TS - 1) / TL_TS, C), 256, smem_tile, e->stream>>>(a, outside ? 1 : 0);
            KCHECK(e);
        } else {
            generic_inside_kernel<<<dim3(gx, C), PLF_TS, smem_in, e->stream>>>(a);
            KCHECK(e);
        }
        generic_site_kernel<<<(a.Sc + 255) / 256, 256, 0, e->stream>>>(a);
        KCHECK(e);
        if (q.sum_ll) {
            wsum_rows_kernel<<<1, 256, 0, e->stream>>>(a.site_ll + s0, w, s0, a.Sc, dsum, e->d_err.as<int>(), 1);
            KCHECK(e);
        }
        if (!outside) {
            zero_lik_rows_kernel<<<(a.Sc + 255) / 256, 256, 0, e->stream>>>(a.site_ll + s0, w, s0, a.Sc, e->d_err.as<int>(),
                                                                            nullptr, 0, nullptr, 0);
            KCHECK(e);
        }
        if (outside) {
            if (q.want_edge) CK(e, cudaMemsetAsync(a.edge_out, 0, sizeof(double) * (size_t)E * a.Sc, e->stream));
            if (q.want_marg) CK(e, cudaMemsetAsync(a.marg_out, 0, sizeof(double) * (size_t)N * n * a.Sc, e->stream));
            if (gm) CK(e, cudaMemsetAsync(a.fe_out, 0, sizeof(double) * (size_t)C * E * n * a.Sc, e->stream));
            if (use_tile) {
                if (tnp == 32) tile_outside_kernel<32><<<(a.Sc + TL_TS - 1) / TL_TS, 128, smem_tile_out, e->stream>>>(a);
                else tile_outside_kernel<64><<<(a.Sc + TL_TS - 1) / TL_TS, 256, smem_tile_out, e->stream>>>(a);
                KCHECK(e);
            } else {
                generic_outside_kernel<<<gx, PLF_TS, smem_out, e->stream>>>(a);
                KCHECK(e);
            }
            zero_lik_rows_kernel<<<(a.Sc + 255) / 256, 256, 0, e->stream>>>(a.site_ll + s0, w, s0, a.Sc, e->d_err.as<int>(),
                                                                            a.edge_out, q.want_edge ? E : 0, a.marg_out, q.want_marg ? N * n : 0);
            KCHECK(e);
            if (gm && E > 0) {
                generic_gmat_kernel<<<dim3(E, C), 256, 0, e->stream>>>(a, dsum + 1);
                KCHECK(e);
            }
            if (q.want_edge && q.sum_edge) {
                wsum_rows_kernel<<<E, 256, 0, e->stream>>>(a.edge_out, w, s0, a.Sc, dsum + 1, e->d_err.as<int>(), 0);
                KCHECK(e);
            }
            if (q.sum_hess) {
                generic_hess_kernel<<<std::min<int>(hgrid, (int)gx), PLF_TS, smem_hess, e->stream>>>(
                    a, ht, e->d_qhi.as<double>(), e->d_cat_rates.as<double>(), w, e->h_Yg.as<double>(), e->h_dFg.as<double>(),
                    e->h_dFk.as<int>(), e->h_part.as<double>(), e->d_err.as<int>());
                KCHECK(e);
                const int nb16 = (E + 15) / 16;
                const int splits = std::max(1, std::min(256, (a.Sc + 4095) / 4096));
                gram_rows_kernel<<<dim3(nb16, nb16, splits), dim3(16, 16), 0, e->stream>>>(a.edge_out, w, s0, E, a.Sc, e->h_gram.as<double>());
                KCHECK(e);
            }
            if (q.want_marg && q.sum_marg) {
                wsum_rows_kernel<<<N * n, 256, 0, e->stream>>>(a.marg_out, w, s0, a.Sc, dsum + 1 + E, e->d_err.as<int>(), 0);
                KCHECK(e);
            }
            if (q.want_edge && q.site_edge) {
                CK(e, cudaStreamSynchronize(e->stream));
                if (copy_site_matrix(e, a.edge_out, E, a.Sc, q.site_edge + (size_t)s0 * E)) return -1;
            }
            if (q.want_marg && q.site_marg) {
                CK(e, cudaStreamSynchronize(e->stream));
                if (copy_site_matrix(e, a.marg_out, N * n, a.Sc, q.site_marg + (size_t)s0 * N * n)) return -1;
            }
        }
    }
    const size_t nsum = gm ? 1 + ngm : 1 + E + (size_t)N * n;
    if (finish_sums(e, dsum, nsum)) return -1;
    if (gm && (run_gmat_adjoint(e, dsum + 1) || copy_gmat_out(e, q))) return -1;
    if (q.sum_hess) {
        /* H = sum of the per-CTA parts - Gram matrix of the per-site derivatives (lower triangle, csr order) */
        sum_rows_kernel<<<(unsigned)(((size_t)E * E + 31) / 32), dim3(32, PLF_ROW_GROUPS), 0, e->stream>>>(e->h_part.as<double>(), hgrid, E * E, e->h_out.as<double>());
        KCHECK(e);
        axpy_kernel<<<(unsigned)(((size_t)E * E + 255) / 256), 256, 0, e->stream>>>(e->h_out.as<double>(), e->h_gram.as<double>(), -1.0, (size_t)E * E);
        KCHECK(e);
        if (finish_sums(e, e->h_out.as<double>(), (size_t)E * E)) return -1;
    }
    std::vector<double> hs; int herr = 0;
    return (read_back(e, q, dsum, nsum, hs, herr) || unpack_sums(e, q, hs, herr)) ? -1 : 0;
}

static int ensure_dm_tables(plf_engine *e, int NB, const double *Fm, int f_zero_rowsum)
{
    if (ensure_program(e)) return -1;
    const int n = e->n, C = e->C, E = e->E, K = e->K;
    const int Ei = (int)e->edge_of_int.size(), Et = (int)e->edge_of_tip.size();
    const size_t slot = dm_slot_doubles_host(NB), W = 8 * (size_t)NB;
    if (!e->dm_valid) {
        ENSURE(e, e->d_dmPf, sizeof(double) * ((size_t)C * Ei * slot + 1));
        ENSURE(e, e->d_dmTPf, sizeof(double) * ((size_t)C * Et * K * W + 1));
        ENSURE(e, e->d_dm_defsf, sizeof(double) * ((size_t)K * W + 1));
        ENSURE(e, e->d_dm_rootf, sizeof(double) * W);
        /* matrices of the outside pass in its consumption order: ops backwards, internal children last to first,
         * P_e then F_e (negative index = second source), all transposed */
        std::vector<int> oidx, otr;
        int depth = 0, sp = 0;
        for (int o = (int)e->ops.size() - 1; o >= 0; o--) {
            const F4Op &op = e->ops[o];
            if (o != (int)e->ops.size() - 1) sp--;
            for (int j = op.nchild - 1; j >= 0; j--) {
                const F4Child &ch = e->children[op.first_child + j];
                if (ch.kind == F4_KIND_TIP) continue;
                oidx.push_back(ch.edge); oidx.push_back(-(ch.edge + 1));
                otr.push_back(1); otr.push_back(1);
                sp++;
                depth = std::max(depth, sp);
            }
        }
        e->dm_out_depth = std::max(depth, 1);
        /* the program in the compact form the kernels stage in shared memory */
        std::vector<int4> ops4(e->ops.size()), ch4(e->children.size());
        for (size_t o = 0; o < e->ops.size(); o++)
            ops4[o] = make_int4(e->ops[o].first_child, e->ops[o].nchild, e->ops[o].code_row, e->ops[o].spill_before);
        for (size_t j = 0; j < e->children.size(); j++)
            ch4[j] = make_int4(e->children[j].kind, e->children[j].mat, e->children[j].code_row, e->children[j].edge);
        ENSURE(e, e->d_dm_ops, sizeof(int4) * (ops4.size() + 1));
        ENSURE(e, e->d_dm_ch, sizeof(int4) * (ch4.size() + 1));
        CK(e, cudaMemcpyAsync(e->d_dm_ops.p, ops4.data(), sizeof(int4) * ops4.size(), cudaMemcpyHostToDevice, e->stream));
        CK(e, cudaMemcpyAsync(e->d_dm_ch.p, ch4.data(), sizeof(int4) * ch4.size(), cudaMemcpyHostToDevice, e->stream));
        ENSURE(e, e->d_dm_oidx, sizeof(int) * (oidx.size() + 1));
        ENSURE(e, e->d_dm_otr, sizeof(int) * (otr.size() + 1));
        std::vector<double> rootf(W, 0.0);
        for (int pos = 0; pos < (int)W; pos++) {
            const int qq = pos / (2 * NB), rem = pos % (2 * NB);
            const int i = 8 * (rem >> 1) + 2 * qq + (rem & 1);
            if (i >= n) continue;
            if (e->root_mode == PLF_ROOT_NONE) rootf[pos] = 1.0;
            else if (e->root_mode == PLF_ROOT_UNIFORM) rootf[pos] = 1.0 / (double)n;
            else rootf[pos] = e->root_vec[i];
        }
        CK(e, cudaMemcpyAsync(e->d_dm_oidx.p, oidx.data(), sizeof(int) * oidx.size(), cudaMemcpyHostToDevice, e->stream));
        CK(e, cudaMemcpyAsync(e->d_dm_otr.p, otr.data(), sizeof(int) * otr.size(), cudaMemcpyHostToDevice, e->stream));
        CK(e, cudaMemcpyAsync(e->d_dm_rootf.p, rootf.data(), sizeof(double) * W, cudaMemcpyHostToDevice, e->stream));
        CK(e, cudaStreamSynchronize(e->stream));
        CK(e, dm_pack(e->d_P.as<double>(), nullptr, e->d_edge_of_int.as<int>(), nullptr, Ei, C, E, n, NB, e->d_dmPf.as<double>(), e->stream));
        e->launches++;
        CK(e, dm_tip_table(e->d_P.as<double>(), e->d_defs.as<double>(), e->d_def_const.as<unsigned char>(), e->d_edge_of_tip.as<int>(),
                           C, E, Et, K, n, NB, 0, e->d_dmTPf.as<double>(), e->stream));
        e->launches++;
        CK(e, dm_tip_table(nullptr, e->d_defs.as<double>(), e->d_def_const.as<unsigned char>(), nullptr,
                           1, E, 1, K, n, NB, 0, e->d_dm_defsf.as<double>(), e->stream));
        e->launches++;
        e->dm_valid = true;
    }
    if (Fm) {
        ENSURE(e, e->d_dm_Of, sizeof(double) * ((size_t)C * 2 * Ei * slot + 1));
        ENSURE(e, e->d_dmTFf, sizeof(double) * ((size_t)C * Et * K * W + 1));
        CK(e, dm_pack(e->d_P.as<double>(), Fm, e->d_dm_oidx.as<int>(), e->d_dm_otr.as<int>(), 2 * Ei, C, E, n, NB, e->d_dm_Of.as<double>(), e->stream));
        e->launches++;
        CK(e, dm_tip_table(Fm, e->d_defs.as<double>(), e->d_def_const.as<unsigned char>(), e->d_edge_of_tip.as<int>(),
                           C, E, Et, K, n, NB, f_zero_rowsum ? 1 : 2, e->d_dmTFf.as<double>(), e->stream));
        e->launches++;
    }
    return 0;
}

/* 16 < n <= 64 (amino-acid, codon models), ll and edge-form queries: the FP64 tensor-pipe kernels of dmma.cu */
static int run_dmma(plf_engine *e, Query &q)
{
    const int n = e->n, C = e->C, E = e->E;
    const int NB = dm_blocks_for(n);
    if (ensure_dm_tables(e, NB, q.want_edge ? q.Fm : nullptr, q.f_zero_rowsum)) return -1;
    const int Ei = (int)e->edge_of_int.size(), Et = (int)e->edge_of_tip.size();
    const int nrows = (int)e->code_row_node.size();

    /* ring slots that fit beside the warps' code tiles */
    const int nops = (int)e->ops.size(), nch = (int)e->children.size();
    int R = 3;      /* measured (2..6): 3 is best by 1-3 %; shared memory not used by the ring is L1 for the tip tables and the slab */
    while (R > 2 && dm_smem_bytes(NB, R, nrows, nops, nch) > 227 * 1024) R--;
    if (dm_smem_bytes(NB, R, nrows, nops, nch) > 227 * 1024) FAIL(e, "tree too large for the tensor-pipe kernels (%d code rows)", nrows);

    /* chunk of sites: the slab of edge vectors (keep mode) is the only large buffer */
    const size_t per_group = q.want_edge ? (size_t)C * Ei * ((size_t)NB * 32 * 16 + 32 * 4) + (size_t)E * 64 : 0;
    size_t free_b = 0, total_b = 0;
    int64_t Sc = e->S;
    /* (the device is only asked for its free memory when the buffers of an earlier query do not already hold the whole alignment) */
    const bool slab_fits = per_group && e->d_dm_slab.cap >= sizeof(double2) * (size_t)C * Ei * ((e->S + 7) / 8) * NB * 32 + 16 &&
                           e->g_edge_out.cap >= sizeof(double) * (size_t)E * e->S && e->S <= ((int64_t)1 << 24);
    if (per_group && !slab_fits) {
        CK(e, cudaMemGetInfo(&free_b, &total_b));
        const size_t have = e->d_dm_slab.cap + e->d_dm_slabmeta.cap + e->g_edge_out.cap;
        const size_t budget = std::min<size_t>((size_t)32 << 30, (free_b + have) / 2);
        const int64_t groups = std::max<int64_t>(DM_TILE / 8, (int64_t)(budget / per_group));
        Sc = std::min<int64_t>(e->S, groups * 8 / DM_TILE * DM_TILE);
    }
    Sc = std::min<int64_t>(Sc, (int64_t)1 << 24);
    const int64_t ngroups_max = (Sc + 7) / 8;

    const int grid_max = e->sm_count;
    ENSURE(e, e->d_dm_stack, sizeof(double2) * (size_t)grid_max * DM_GROUPS * std::max(1, std::max(e->stack_depth, q.want_edge ? 2 * e->dm_out_depth : 0)) * NB * 32);
    ENSURE(e, e->d_dm_stackmeta, sizeof(int) * (size_t)grid_max * DM_GROUPS * std::max(1, std::max(e->stack_depth, q.want_edge ? 4 * e->dm_out_depth : 0)) * 32);
    ENSURE(e, e->g_cat_lh, sizeof(double) * (size_t)C * Sc);
    ENSURE(e, e->g_cat_k, sizeof(int) * (size_t)C * Sc);
    ENSURE(e, e->g_site_m, sizeof(double) * Sc);
    ENSURE(e, e->g_site_k, sizeof(int) * Sc);
    if (prepare_sums(e, 1 + E)) return -1;
    if (q.want_edge) {
        ENSURE(e, e->d_dm_slab, sizeof(double2) * (size_t)C * Ei * ngroups_max * NB * 32 + 16);
        ENSURE(e, e->d_dm_slabmeta, sizeof(int) * (size_t)C * Ei * ngroups_max * 32 + 16);
        ENSURE(e, e->g_edge_out, sizeof(double) * (size_t)E * Sc);
    }
    double *dsum = e->d_sum.as<double>();
    CK(e, cudaMemsetAsync(dsum, 0, sizeof(double) * (1 + E), e->stream));

    DmArgs a;
    memset(&a, 0, sizeof(a));
    a.n = n; a.C = C; a.K = e->K;
    a.nops = nops; a.nchildren = nch; a.ops4 = e->d_dm_ops.as<int4>(); a.ch4 = e->d_dm_ch.as<int4>();
    a.Ei = Ei; a.Et = Et; a.nrows = nrows; a.code_row_node = e->d_code_row_node.as<int>();
    a.codes = e->d_codes.as<unsigned char>(); a.S = e->S;
    a.def_const = e->d_def_const.as<unsigned char>(); a.defsf = e->d_dm_defsf.as<double>();
    a.Pf = e->d_dmPf.as<double>(); a.TPf = e->d_dmTPf.as<double>(); a.rootf = e->d_dm_rootf.as<double>();
    a.root_const_ok = (e->root_mode == PLF_ROOT_UNIFORM || e->root_mode == PLF_ROOT_EQUILIBRIUM) ? 1 : 0;
    a.cat_lh = e->g_cat_lh.as<double>(); a.cat_k = e->g_cat_k.as<int>();
    a.R = R;
    a.stack = e->d_dm_stack.as<double2>(); a.stack_meta = e->d_dm_stackmeta.as<int>();
    a.Of = e->d_dm_Of.as<double>(); a.TFf = e->d_dmTFf.as<double>();
    a.cat_prior = e->d_cat_prior.as<double>();
    a.site_m = e->g_site_m.as<double>(); a.site_k = e->g_site_k.as<int>();
    a.edge_mask = q.edge_mask_h ? e->d_mask.as<unsigned char>() : nullptr;
    a.f_zero_rowsum = q.f_zero_rowsum;
    a.edge_out = q.want_edge ? e->g_edge_out.as<double>() : nullptr;

    /* generic_site_kernel combines the categories */
    GenericArgs ga;
    memset(&ga, 0, sizeof(ga));
    ga.C = C; ga.cat_prior = a.cat_prior; ga.cat_lh = a.cat_lh; ga.cat_k = a.cat_k;
    ga.site_m = e->g_site_m.as<double>(); ga.site_k = e->g_site_k.as<int>(); ga.site_ll = e->d_site_ll.as<double>();

    const double *w = e->have_w ? e->d_site_w.as<double>() : nullptr;
    {
        char nm[96];
        snprintf(nm, sizeof nm, q.want_edge ? "dm_inside_kernel<%d,16,1> + dm_outside_kernel<%d,16,1>" : "dm_inside_kernel<%d,16,1>", NB, NB);
        e->last_kernel = nm;
    }
    CK(e, cudaEventRecord(e->ev[3], e->stream));
    for (int64_t s0 = 0; s0 < e->S; s0 += Sc) {
        a.s0 = s0; a.Sc = (int)std::min<int64_t>(Sc, e->S - s0);
        a.ngroups = (a.Sc + 7) / 8;
        dm_tiling(a.ngroups, C, grid_max, &a.tiles_full, &a.tail_gs, &a.ntiles);
        a.slab = q.want_edge ? e->d_dm_slab.as<double2>() : nullptr;
        a.slab_meta = q.want_edge ? e->d_dm_slabmeta.as<int>() : nullptr;
        a.stack_depth = std::max(1, e->stack_depth);
        const long long items = (long long)a.ntiles * C;
        CK(e, dm_launch_inside(a, NB, (int)std::min<long long>(grid_max, items), e->stream));
        e->launches++;
        ga.s0 = s0; ga.Sc = a.Sc;
        generic_site_kernel<<<(a.Sc + 255) / 256, 256, 0, e->stream>>>(ga);
        KCHECK(e);
        if (q.sum_ll) {
            wsum_rows_kernel<<<1, 256, 0, e->stream>>>(ga.site_ll + s0, w, s0, a.Sc, dsum, e->d_err.as<int>(), 1);
            KCHECK(e);
        }
        if (!q.want_edge) {
            zero_lik_rows_kernel<<<(a.Sc + 255) / 256, 256, 0, e->stream>>>(ga.site_ll + s0, w, s0, a.Sc, e->d_err.as<int>(),
                                                                            nullptr, 0, nullptr, 0);
            KCHECK(e);
        }
        if (q.want_edge) {
            CK(e, cudaMemsetAsync(a.edge_out, 0, sizeof(double) * (size_t)E * a.Sc, e->stream));
            a.stack_depth = e->dm_out_depth;
            dm_tiling(a.ngroups, 1, grid_max, &a.tiles_full, &a.tail_gs, &a.ntiles);
            CK(e, dm_launch_outside(a, NB, std::min(grid_max, a.ntiles), e->stream));
            e->launches++;
            zero_lik_rows_kernel<<<(a.Sc + 255) / 256, 256, 0, e->stream>>>(ga.site_ll + s0, w, s0, a.Sc, e->d_err.as<int>(),
                                                                            a.edge_out, E, nullptr, 0);
            KCHECK(e);
            if (q.sum_edge) {
                wsum_rows_kernel<<<E, 256, 0, e->stream>>>(a.edge_out, w, s0, a.Sc, dsum + 1, e->d_err.as<int>(), 0);
                KCHECK(e);
            }
            if (q.site_edge) {
                CK(e, cudaStreamSynchronize(e->stream));
                if (copy_site_matrix(e, a.edge_out, E, a.Sc, q.site_edge + (size_t)s0 * E)) return -1;
            }
        }
    }
    CK(e, cudaEventRecord(e->ev[4], e->stream));
    e->kernel_timed = true;
    const size_t nsum = 1 + E;
    if (finish_sums(e, dsum, nsum)) return -1;
    std::vector<double> hs; int herr = 0;
    return (read_back(e, q, dsum, nsum, hs, herr) || unpack_sums(e, q, hs, herr)) ? -1 : 0;
}

enum class QueryPath { fused, fused_windows, dmma, tile, generic };

/* The kernels a query runs.  An upload in flight is resolved here, before the tree program is built, unless the query
 * takes the single-window fused path: only run_fused overlaps an upload, and it repeats the query when the upload
 * changes which nodes carry data. */
static int choose_path(plf_engine *e, const Query &q, QueryPath &path)
{
    const bool generic_only = e->path == PLF_PATH_GENERIC;
    /* the edge matrices need the whole site likelihood: no category windows (n = 4 with C > 4 goes to the generic
     * path); per-site marginals of a huge alignment: the generic path works in chunks of sites */
    bool fused = e->n == 4 && e->C <= 16 && e->code_bytes == 1 && e->K <= 256 && e->max_degree <= F4_MAXD && !generic_only &&
                 !q.sum_hess && !(q.want_gmat && e->C > 4) &&
                 !(q.want_marg && q.site_marg && (size_t)e->N * 4 * e->S * sizeof(double) > ((size_t)32 << 30));
    const bool windows = e->C > 4 && !q.want_gmat;
    const bool overlap = fused && !windows && e->node_has_data_h.size() == (size_t)e->N;
    if (!overlap && resolve_pending(e)) return -1;
    if (fused) {
        if (ensure_program(e)) return -1;
        fused = fused_fits(e, q.want_edge || q.want_marg || q.want_gmat);
    }
    if (!fused && resolve_pending(e)) return -1;
    if (e->path == PLF_PATH_FUSED4 && !fused) FAIL(e, "the fused 4-state path does not apply to this query");
    if (fused) path = windows ? QueryPath::fused_windows : QueryPath::fused;
    else if (!generic_only && !q.sum_hess && !q.want_gmat && !q.want_marg && dm_blocks_for(e->n) != 0 && e->code_bytes == 1 &&
             e->K <= 256)
        path = QueryPath::dmma;
    else if (e->n > 16 && e->n <= TL_NP && !getenv("PLF_NO_TILE") && !q.sum_hess && !q.want_gmat) path = QueryPath::tile;
    else path = QueryPath::generic;
    return 0;
}

/* common driver: matrices, path selection, timing.  Returns 1 when the query has to be repeated. */
static int run_query_once(plf_engine *e, Query &q, bool need_D, const double *l_hi, const double *l_lo, int kind)
{
    if (e->S == 0 || e->n == 0 || e->N == 0) FAIL(e, "engine is not fully configured (tree, model and data are required)");
    CK(e, cudaSetDevice(e->device));
    if (q.edge_mask_h) {
        ENSURE(e, e->d_mask, e->E);
        CK(e, cudaMemcpyAsync(e->d_mask.p, q.edge_mask_h, e->E, cudaMemcpyHostToDevice, e->stream));
    }
    QueryPath path;
    if (choose_path(e, q, path)) return -1;
    const bool fused = path == QueryPath::fused || path == QueryPath::fused_windows;
    CK(e, cudaEventRecord(e->ev[0], e->stream));
    if (ensure_matrices(e, need_D)) return -1;
    int f_mode = 2;
    if (need_D) { q.Fm = e->d_D.as<double>(); q.f_zero_rowsum = 1; f_mode = 1; }
    if (l_hi) {
        if (upload_L(e, l_hi, l_lo)) return -1;
        ENSURE(e, e->d_F, sizeof(double) * (size_t)e->C * e->E * e->n * e->n);
        if (run_expm(e, nullptr, nullptr, e->d_F.as<double>(), kind == PLF_KIND_TRANS ? 1 : 0,
                     q.edge_mask_h ? e->d_mask.as<unsigned char>() : nullptr, e->d_lhi.as<double>(), e->d_llo.as<double>())) return -1;
        q.Fm = e->d_F.as<double>(); q.f_zero_rowsum = 0; f_mode = 2;
    }
    if (fused && ensure_tip_tables(e, q.want_edge ? q.Fm : nullptr, f_mode, q.want_marg)) return -1;
    CK(e, cudaEventRecord(e->ev[1], e->stream));
    e->kernel_timed = false;
    e->ms_kernel_override = -1.f;
    int rc;
    switch (path) {
    case QueryPath::fused: rc = run_fused(e, q); break;
    case QueryPath::fused_windows: rc = run_fused_windows(e, q); break;
    case QueryPath::dmma: rc = run_dmma(e, q); break;
    default: rc = run_generic(e, q, path == QueryPath::tile); break;
    }
    if (rc) return rc;
    cudaEventElapsedTime(&e->ms_mat, e->ev[0], e->ev[1]);
    cudaEventElapsedTime(&e->ms_sites, e->ev[1], e->ev[2]);
    e->ms_kernel = 0.f;
    if (e->kernel_timed) cudaEventElapsedTime(&e->ms_kernel, e->ev[3], e->ev[4]);
    if (e->ms_kernel_override >= 0.f) e->ms_kernel = e->ms_kernel_override;
    return 0;
}

static int run_query(plf_engine *e, Query &q, bool need_D, const double *l_hi, const double *l_lo, int kind)
{
    int rc = run_query_once(e, q, need_D, l_hi, l_lo, kind);
    if (rc == 1) rc = run_query_once(e, q, need_D, l_hi, l_lo, kind);
    return rc;
}

extern "C" int plf_ll(plf_engine *e, double *site_ll, double *sum)
{
    if (!e) return -1;
    Query q;
    q.site_ll = site_ll; q.sum_ll = sum;
    return run_query(e, q, false, nullptr, nullptr, 0);
}

extern "C" int plf_deriv(plf_engine *e, const unsigned char *edge_mask, double *site_ll, double *sum_ll,
                         double *site_deriv, double *sum_deriv)
{
    if (!e) return -1;
    Query q;
    q.want_edge = true; q.edge_mask_h = edge_mask;
    q.site_ll = site_ll; q.sum_ll = sum_ll; q.site_edge = site_deriv; q.sum_edge = sum_deriv;
    return run_query(e, q, true, nullptr, nullptr, 0);
}

extern "C" int plf_hess(plf_engine *e, double *sum_ll, double *sum_deriv, double *sum_hess)
{
    if (!e) return -1;
    if (!sum_hess) FAIL(e, "plf_hess: sum_hess is required");
    Query q;
    q.want_edge = true;
    q.sum_ll = sum_ll; q.sum_edge = sum_deriv; q.sum_hess = sum_hess;
    std::vector<double> tmp;
    if (!q.sum_edge) { tmp.resize(e->E > 0 ? e->E : 1); q.sum_edge = tmp.data(); }
    return run_query(e, q, true, nullptr, nullptr, 0);
}

extern "C" int plf_marginal(plf_engine *e, double *site_marg, double *sum_marg)
{
    if (!e) return -1;
    Query q;
    q.want_marg = true; q.site_marg = site_marg; q.sum_marg = sum_marg;
    return run_query(e, q, false, nullptr, nullptr, 0);
}

extern "C" int plf_edge_expect(plf_engine *e, int kind, const double *l_hi, const double *l_lo,
                               const unsigned char *edge_mask, double *site_out, double *sum_out)
{
    if (!e) return -1;
    if (kind != PLF_KIND_DWELL && kind != PLF_KIND_TRANS) FAIL(e, "plf_edge_expect: invalid kind %d", kind);
    if (!l_hi) FAIL(e, "plf_edge_expect: l_hi is required");
    Query q;
    q.want_edge = true; q.edge_mask_h = edge_mask; q.site_edge = site_out; q.sum_edge = sum_out;
    return run_query(e, q, false, l_hi, l_lo, kind);
}

extern "C" int plf_edge_expect_all(plf_engine *e, double *sum_ll, double *dwell, double *trans)
{
    if (!e) return -1;
    Query q;
    q.want_gmat = true; q.sum_ll = sum_ll; q.dwell_out = dwell; q.trans_out = trans;
    return run_query(e, q, false, nullptr, nullptr, 0);
}

extern "C" int plf_get_transition_matrices(plf_engine *e, double *p_out)
{
    if (!e) return -1;
    if (e->n == 0) FAIL(e, "model not set");
    CK(e, cudaSetDevice(e->device));
    if (ensure_matrices(e, false)) return -1;
    CK(e, cudaMemcpyAsync(p_out, e->d_P.p, sizeof(double) * (size_t)e->C * e->E * e->n * e->n, cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    return 0;
}

extern "C" int plf_get_derivative_matrices(plf_engine *e, double *d_out)
{
    if (!e) return -1;
    if (e->n == 0) FAIL(e, "model not set");
    CK(e, cudaSetDevice(e->device));
    if (ensure_matrices(e, true)) return -1;
    CK(e, cudaMemcpyAsync(d_out, e->d_D.p, sizeof(double) * (size_t)e->C * e->E * e->n * e->n, cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    return 0;
}

extern "C" int plf_get_frechet_matrices(plf_engine *e, const double *l_hi, const double *l_lo, double *f_out)
{
    if (!e) return -1;
    if (e->n == 0) FAIL(e, "model not set");
    CK(e, cudaSetDevice(e->device));
    if (upload_L(e, l_hi, l_lo)) return -1;
    ENSURE(e, e->d_F, sizeof(double) * (size_t)e->C * e->E * e->n * e->n);
    if (run_expm(e, nullptr, nullptr, e->d_F.as<double>(), 0, nullptr, e->d_lhi.as<double>(), e->d_llo.as<double>())) return -1;
    CK(e, cudaMemcpyAsync(f_out, e->d_F.p, sizeof(double) * (size_t)e->C * e->E * e->n * e->n, cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    return 0;
}

/* ------------------------------------------------------------------ */
/* certified mode                                                      */
/* ------------------------------------------------------------------ */

/* v (1 - d) rounded down / v (1 + d) rounded up, for v >= 0 */
static double cert_lo_h(double v, double d) { return v <= 0.0 ? 0.0 : std::nextafter(v * (1.0 - d), -INFINITY); }
static double cert_hi_h(double v, double d) { return v <= 0.0 ? 0.0 : std::nextafter(v * (1.0 + d), INFINITY); }

/* Enclosures of the transition matrices (and, with D, of r_c Q P_e) on the device, and those of the root weights and
 * the category priors in c_small = [root_lo | root_hi | prior_lo | prior_hi] (exact when they are the user's own numbers) */
static int cert_prepare(plf_engine *e, double delta_rate, double delta_q, bool with_D)
{
    const int n = e->n, C = e->C, E = e->E;
    const size_t nn = (size_t)n * n;
    ENSURE(e, e->c_Plo, sizeof(double) * C * E * nn + 8);
    ENSURE(e, e->c_Phi, sizeof(double) * C * E * nn + 8);
    ENSURE(e, e->c_ws, sizeof(double) * C * E * 8 * nn + 8);
    if (with_D) {
        ENSURE(e, e->c_Dlo, sizeof(double) * C * E * nn + 8);
        ENSURE(e, e->c_Dhi, sizeof(double) * C * E * nn + 8);
    }
    if (E > 0) {
        cert_expm_kernel<<<dim3(E, C), 128, 0, e->stream>>>(n, E, C, e->d_qhi.as<double>(), e->d_qlo.as<double>(), e->d_edge_rates.as<double>(),
                                                            e->d_cat_rates.as<double>(), delta_rate, delta_q, e->c_ws.as<double>(),
                                                            e->c_Plo.as<double>(), e->c_Phi.as<double>(),
                                                            with_D ? e->c_Dlo.as<double>() : nullptr, with_D ? e->c_Dhi.as<double>() : nullptr);
        KCHECK(e);
    }
    std::vector<double> small(2 * (size_t)n + 2 * (size_t)C);
    double *rlo = small.data(), *rhi = rlo + n, *plo = rhi + n, *phi = plo + C;
    for (int i = 0; i < n; i++) {
        if (e->root_mode == PLF_ROOT_NONE) { rlo[i] = rhi[i] = 1.0; }
        else if (e->root_mode == PLF_ROOT_UNIFORM) { rlo[i] = std::nextafter(1.0 / n, 0.0); rhi[i] = std::nextafter(1.0 / n, 1.0); }
        else if (e->root_mode == PLF_ROOT_CUSTOM) { rlo[i] = rhi[i] = e->root_vec[i]; }
        else { rlo[i] = cert_lo_h(e->root_vec[i], delta_rate); rhi[i] = cert_hi_h(e->root_vec[i], delta_rate); }
    }
    for (int c = 0; c < C; c++) { plo[c] = cert_lo_h(e->cat_prior[c], delta_q); phi[c] = cert_hi_h(e->cat_prior[c], delta_q); }
    ENSURE(e, e->c_small, sizeof(double) * small.size());
    CK(e, cudaMemcpyAsync(e->c_small.p, small.data(), sizeof(double) * small.size(), cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    return 0;
}

extern "C" int plf_ll_certified(plf_engine *e, double delta_rate, double delta_q, double *site_lo, double *site_hi,
                                double *sum_lo, double *sum_hi)
{
    if (!e) return -1;
    if (e->S == 0 || e->n == 0 || e->N == 0) FAIL(e, "engine is not fully configured (tree, model and data are required)");
    if (!(delta_rate >= 0.0) || !(delta_q >= 0.0) || delta_rate > 1e-3 || delta_q > 1e-3) FAIL(e, "plf_ll_certified: bad input uncertainties");
    CK(e, cudaSetDevice(e->device));
    if (resolve_pending(e)) return -1;
    const int n = e->n, C = e->C, N = e->N, E = e->E;
    if (cert_prepare(e, delta_rate, delta_q, false)) return -1;

    const size_t per_site = (size_t)C * ((size_t)2 * N * n * 8 + (size_t)N * 5 + 24) + 16;
    size_t free_b = 0, total_b = 0;
    CK(e, cudaMemGetInfo(&free_b, &total_b));
    const size_t budget = std::min<size_t>((size_t)24 << 30, free_b / 2 + e->g_Lg.cap + e->g_Fg.cap);
    int64_t Sc = std::max<int64_t>(CERT_TS, std::min<int64_t>(e->S, (int64_t)(budget / per_site)));
    Sc = std::min<int64_t>(Sc, 1 << 20);
    if (Sc < e->S) Sc = (Sc / CERT_TS) * CERT_TS;
    ENSURE(e, e->g_Lg, sizeof(double) * (size_t)C * N * n * Sc);
    ENSURE(e, e->g_Fg, sizeof(double) * (size_t)C * N * n * Sc);
    ENSURE(e, e->g_Kg, sizeof(int) * (size_t)C * N * Sc);
    ENSURE(e, e->g_Cg, (size_t)C * N * Sc);
    ENSURE(e, e->g_cat_lh, sizeof(double) * (size_t)C * Sc);
    ENSURE(e, e->c_cat_hi, sizeof(double) * (size_t)C * Sc);
    ENSURE(e, e->g_cat_k, sizeof(int) * (size_t)C * Sc);
    ENSURE(e, e->c_site_lo, sizeof(double) * e->S);
    ENSURE(e, e->c_site_hi, sizeof(double) * e->S);

    CertArgs a;
    memset(&a, 0, sizeof(a));
    a.t.N = N; a.t.E = E; a.t.root = e->root;
    a.t.indptr = e->d_indptr.as<int>(); a.t.indices = e->d_indices.as<int>(); a.t.preorder = e->d_preorder.as<int>();
    a.t.node_has_data = e->d_node_has_data.as<unsigned char>();
    a.n = n; a.C = C; a.K = e->K; a.S = e->S;
    a.codes = e->d_codes.p; a.code_bytes = e->code_bytes;
    a.defs = e->d_defs.as<double>(); a.def_const = e->d_def_const.as<unsigned char>();
    a.Plo = e->c_Plo.as<double>(); a.Phi = e->c_Phi.as<double>();
    a.root_mode = e->root_mode;
    a.root_lo = e->c_small.as<double>(); a.root_hi = a.root_lo + n; a.prior_lo = a.root_hi + n; a.prior_hi = a.prior_lo + C;
    a.Llo = e->g_Lg.as<double>(); a.Lhi = e->g_Fg.as<double>(); a.Kg = e->g_Kg.as<int>(); a.Cg = e->g_Cg.as<unsigned char>();
    a.cat_lo = e->g_cat_lh.as<double>(); a.cat_hi = e->c_cat_hi.as<double>(); a.cat_k = e->g_cat_k.as<int>();
    a.site_lo = e->c_site_lo.as<double>(); a.site_hi = e->c_site_hi.as<double>();
    const size_t smem = sizeof(double) * 4 * n * CERT_TS;
    if (smem > 227 * 1024) FAIL(e, "state count %d is too large for the certified kernels", n);
    if (smem > 48 * 1024) CK(e, cudaFuncSetAttribute(cert_inside_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    e->last_kernel = "cert_expm_kernel + cert_inside_kernel";
    for (int64_t s0 = 0; s0 < e->S; s0 += Sc) {
        a.s0 = s0; a.Sc = (int)std::min<int64_t>(Sc, e->S - s0);
        cert_inside_kernel<<<dim3((a.Sc + CERT_TS - 1) / CERT_TS, C), CERT_TS, smem, e->stream>>>(a);
        KCHECK(e);
        cert_site_kernel<<<(a.Sc + 255) / 256, 256, 0, e->stream>>>(a);
        KCHECK(e);
    }
    std::vector<double> lo_h, hi_h;
    double *lo_p = site_lo, *hi_p = site_hi;
    if (!lo_p) { lo_h.resize(e->S); lo_p = lo_h.data(); }
    if (!hi_p) { hi_h.resize(e->S); hi_p = hi_h.data(); }
    CK(e, cudaMemcpyAsync(lo_p, e->c_site_lo.p, sizeof(double) * e->S, cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaMemcpyAsync(hi_p, e->c_site_hi.p, sizeof(double) * e->S, cudaMemcpyDeviceToHost, e->stream));
    std::vector<double> w_h;
    if (e->have_w && (sum_lo || sum_hi)) {
        w_h.resize(e->S);
        CK(e, cudaMemcpyAsync(w_h.data(), e->d_site_w.p, sizeof(double) * e->S, cudaMemcpyDeviceToHost, e->stream));
    }
    CK(e, cudaStreamSynchronize(e->stream));
    if (sum_lo || sum_hi) {
        /* weighted sums of the enclosures with the host's rounding mode set for each bound */
        const int old = fegetround();
        volatile double acc_lo = 0.0, acc_hi = 0.0;
        bool bad = false;
        fesetround(FE_DOWNWARD);
        for (int64_t i = 0; i < e->S; i++) {
            const double w = w_h.empty() ? 1.0 : w_h[i];
            if (w == 0.0) continue;
            volatile double term = w * (w > 0.0 ? lo_p[i] : hi_p[i]);
            if (!std::isfinite(term)) bad = true;
            acc_lo = acc_lo + term;
        }
        fesetround(FE_UPWARD);
        for (int64_t i = 0; i < e->S; i++) {
            const double w = w_h.empty() ? 1.0 : w_h[i];
            if (w == 0.0) continue;
            volatile double term = w * (w > 0.0 ? hi_p[i] : lo_p[i]);
            if (!std::isfinite(term)) bad = true;
            acc_hi = acc_hi + term;
        }
        fesetround(old);
        if (bad) FAIL(e, "a site with non-zero weight has zero likelihood");
        if (sum_lo) *sum_lo = acc_lo;
        if (sum_hi) *sum_hi = acc_hi;
    }
    return 0;
}

/* the checks every certified outside query makes before it launches anything */
static int cert_check(plf_engine *e, const char *what, double delta_rate, double delta_q)
{
    if (e->S == 0 || e->n == 0 || e->N == 0) FAIL(e, "engine is not fully configured (tree, model and data are required)");
    if (!(delta_rate >= 0.0) || !(delta_q >= 0.0) || delta_rate > 1e-3 || delta_q > 1e-3) FAIL(e, "%s: bad input uncertainties", what);
    if (sizeof(double) * 6 * e->n * CERT_TS > 227 * 1024) FAIL(e, "state count %d is too large for the certified kernels", e->n);
    return 0;
}

enum CertOutside { CERT_DERIV, CERT_EXPECT, CERT_MARGINAL };

/*
 * The site passes of the certified outside queries, after cert_prepare (and, for the edge forms, the edge matrices in
 * c_Dlo / c_Dhi and the mask in d_mask): per chunk the inside pass, the site likelihood enclosure, the outside pass,
 * the per-site columns (edges, or node x state for CERT_MARGINAL) and their group sums; then the totals and the
 * read-back.  Per-site output [S][cols], sums [cols].
 */
static int cert_outside_query(plf_engine *e, CertOutside what, const unsigned char *edge_mask, double *site_lo, double *site_hi,
                              double *sum_lo, double *sum_hi)
{
    const int n = e->n, C = e->C, N = e->N, E = e->E;
    const bool edges = what != CERT_MARGINAL;
    const int cols = edges ? E : N * n;
    const size_t smem_in = sizeof(double) * 4 * n * CERT_TS, smem_out = sizeof(double) * 6 * n * CERT_TS;
    /* inside and outside vectors, edge forms, the site likelihood enclosure and the per-site output of a chunk */
    const size_t per_site = (size_t)C * ((size_t)4 * N * n * 8 + (size_t)N * 9 + (edges ? (size_t)E * 20 : 0) + 24) + (size_t)cols * 16 + 24;
    size_t free_b = 0, total_b = 0;
    CK(e, cudaMemGetInfo(&free_b, &total_b));
    const size_t held = e->g_Lg.cap + e->g_Fg.cap + e->c_Flo.cap + e->c_Fhi.cap + e->c_xlo.cap + e->c_xhi.cap + e->c_olo.cap + e->c_ohi.cap;
    const size_t budget = std::min<size_t>((size_t)24 << 30, free_b / 2 + held);
    int64_t Sc = std::max<int64_t>(CERT_GROUP, std::min<int64_t>(e->S, (int64_t)(budget / per_site)));
    Sc = std::min<int64_t>(Sc, 1 << 20);
    if (Sc < e->S) Sc = (Sc / CERT_GROUP) * CERT_GROUP;
    Sc = std::min<int64_t>(Sc, e->S);
    ENSURE(e, e->g_Lg, sizeof(double) * (size_t)C * N * n * Sc);
    ENSURE(e, e->g_Fg, sizeof(double) * (size_t)C * N * n * Sc);
    ENSURE(e, e->g_Kg, sizeof(int) * (size_t)C * N * Sc);
    ENSURE(e, e->g_Cg, (size_t)C * N * Sc);
    ENSURE(e, e->g_cat_lh, sizeof(double) * (size_t)C * Sc);
    ENSURE(e, e->c_cat_hi, sizeof(double) * (size_t)C * Sc);
    ENSURE(e, e->g_cat_k, sizeof(int) * (size_t)C * Sc);
    ENSURE(e, e->c_site_lo, sizeof(double) * e->S);
    ENSURE(e, e->c_site_hi, sizeof(double) * e->S);
    ENSURE(e, e->c_Flo, sizeof(double) * (size_t)C * N * n * Sc);
    ENSURE(e, e->c_Fhi, sizeof(double) * (size_t)C * N * n * Sc);
    ENSURE(e, e->c_FK, sizeof(int) * (size_t)C * N * Sc);
    if (edges) {
        ENSURE(e, e->c_xlo, sizeof(double) * (size_t)C * E * Sc);
        ENSURE(e, e->c_xhi, sizeof(double) * (size_t)C * E * Sc);
        ENSURE(e, e->c_xk, sizeof(int) * (size_t)C * E * Sc);
    }
    ENSURE(e, e->c_mlo, sizeof(double) * Sc);
    ENSURE(e, e->c_mhi, sizeof(double) * Sc);
    ENSURE(e, e->c_mk, sizeof(int) * Sc);
    ENSURE(e, e->c_olo, sizeof(double) * (size_t)cols * Sc);
    ENSURE(e, e->c_ohi, sizeof(double) * (size_t)cols * Sc);
    const int64_t groups = (e->S + CERT_GROUP - 1) / CERT_GROUP;
    ENSURE(e, e->c_part, sizeof(double) * 2 * (size_t)groups * cols);
    ENSURE(e, e->c_sums, sizeof(double) * 2 * (size_t)cols);
    ENSURE(e, e->c_err, sizeof(int));
    CK(e, cudaMemsetAsync(e->c_err.p, 0, sizeof(int), e->stream));

    CertArgs a;
    memset(&a, 0, sizeof(a));
    a.t.N = N; a.t.E = E; a.t.root = e->root;
    a.t.indptr = e->d_indptr.as<int>(); a.t.indices = e->d_indices.as<int>(); a.t.preorder = e->d_preorder.as<int>();
    a.t.node_has_data = e->d_node_has_data.as<unsigned char>();
    a.n = n; a.C = C; a.K = e->K; a.S = e->S;
    a.codes = e->d_codes.p; a.code_bytes = e->code_bytes;
    a.defs = e->d_defs.as<double>(); a.def_const = e->d_def_const.as<unsigned char>();
    a.Plo = e->c_Plo.as<double>(); a.Phi = e->c_Phi.as<double>();
    a.root_mode = e->root_mode;
    a.root_lo = e->c_small.as<double>(); a.root_hi = a.root_lo + n; a.prior_lo = a.root_hi + n; a.prior_hi = a.prior_lo + C;
    a.Llo = e->g_Lg.as<double>(); a.Lhi = e->g_Fg.as<double>(); a.Kg = e->g_Kg.as<int>(); a.Cg = e->g_Cg.as<unsigned char>();
    a.cat_lo = e->g_cat_lh.as<double>(); a.cat_hi = e->c_cat_hi.as<double>(); a.cat_k = e->g_cat_k.as<int>();
    a.site_lo = e->c_site_lo.as<double>(); a.site_hi = e->c_site_hi.as<double>();
    a.site_mlo = e->c_mlo.as<double>(); a.site_mhi = e->c_mhi.as<double>(); a.site_k = e->c_mk.as<int>();
    if (edges) {
        a.Dlo = e->c_Dlo.as<double>(); a.Dhi = e->c_Dhi.as<double>();
        a.xlo = e->c_xlo.as<double>(); a.xhi = e->c_xhi.as<double>(); a.xk = e->c_xk.as<int>();
        a.edge_mask = edge_mask ? e->d_mask.as<unsigned char>() : nullptr;
    }
    a.deriv = what == CERT_DERIV;
    a.marg = what == CERT_MARGINAL;
    a.cat_rate = e->d_cat_rates.as<double>();
    a.Flo = e->c_Flo.as<double>(); a.Fhi = e->c_Fhi.as<double>(); a.FK = e->c_FK.as<int>();
    a.site_w = e->have_w ? e->d_site_w.as<double>() : nullptr;
    a.out_lo = e->c_olo.as<double>(); a.out_hi = e->c_ohi.as<double>();
    a.err = e->c_err.as<int>();
    if (smem_in > 48 * 1024) CK(e, cudaFuncSetAttribute(cert_inside_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_in));
    if (smem_out > 48 * 1024) CK(e, cudaFuncSetAttribute(cert_outside_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_out));
    const bool sums = sum_lo || sum_hi;
    double *part_lo = e->c_part.as<double>(), *part_hi = part_lo + (size_t)groups * cols;
    for (int64_t s0 = 0; s0 < e->S; s0 += Sc) {
        a.s0 = s0; a.Sc = (int)std::min<int64_t>(Sc, e->S - s0);
        const unsigned tiles = (unsigned)((a.Sc + CERT_TS - 1) / CERT_TS);
        cert_inside_kernel<<<dim3(tiles, C), CERT_TS, smem_in, e->stream>>>(a);
        KCHECK(e);
        cert_site_kernel<<<(a.Sc + 255) / 256, 256, 0, e->stream>>>(a);
        KCHECK(e);
        cert_outside_kernel<<<dim3(tiles, C), CERT_TS, smem_out, e->stream>>>(a);
        KCHECK(e);
        for (int e0 = 0; e0 < cols; e0 += 65535) {          /* the grid's y extent */
            const dim3 site_grid((a.Sc + 127) / 128, std::min(cols - e0, 65535)), group_grid((a.Sc + CERT_GROUP - 1) / CERT_GROUP, site_grid.y);
            if (edges) cert_deriv_site_kernel<<<site_grid, 128, 0, e->stream>>>(a, a.xlo, a.xhi, a.xk, E, 1, e0);
            else cert_deriv_site_kernel<<<site_grid, 128, 0, e->stream>>>(a, a.Flo, a.Fhi, a.FK, cols, n, e0);
            KCHECK(e);
            if (sums) {
                cert_deriv_group_sum_kernel<<<group_grid, 32, 0, e->stream>>>(a, cols, e0, part_lo, part_hi);
                KCHECK(e);
            }
        }
        /* per-site outputs of the chunk, [cols][Sc] on the device -> rows s0.. of [S][cols] on the host */
        if (site_lo && copy_site_matrix(e, a.out_lo, cols, a.Sc, site_lo + (size_t)s0 * cols)) return -1;
        if (site_hi && copy_site_matrix(e, a.out_hi, cols, a.Sc, site_hi + (size_t)s0 * cols)) return -1;
    }
    double *d_sums = e->c_sums.as<double>();
    if (sums) {
        cert_deriv_total_kernel<<<(cols + 127) / 128, 128, 0, e->stream>>>(part_lo, part_hi, (int)groups, cols, d_sums, d_sums + cols);
        KCHECK(e);
    }
    std::vector<double> sums_h(sums ? 2 * (size_t)cols : 0);
    int err = 0;
    if (sums) CK(e, cudaMemcpyAsync(sums_h.data(), d_sums, sizeof(double) * 2 * cols, cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaMemcpyAsync(&err, e->c_err.p, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    if (sums) {
        if (err & 1) FAIL(e, "a site with non-zero weight has zero likelihood");
        if (sum_lo) memcpy(sum_lo, sums_h.data(), sizeof(double) * cols);
        if (sum_hi) memcpy(sum_hi, sums_h.data() + cols, sizeof(double) * cols);
    }
    return 0;
}

extern "C" int plf_deriv_certified(plf_engine *e, double delta_rate, double delta_q, const unsigned char *edge_mask,
                                   double *site_lo, double *site_hi, double *sum_lo, double *sum_hi)
{
    if (!e) return -1;
    if (cert_check(e, "plf_deriv_certified", delta_rate, delta_q)) return -1;
    CK(e, cudaSetDevice(e->device));
    if (resolve_pending(e)) return -1;
    if (e->E == 0) return 0;
    if (cert_prepare(e, delta_rate, delta_q, true)) return -1;
    ENSURE(e, e->d_mask, (size_t)e->E);
    if (edge_mask) CK(e, cudaMemcpyAsync(e->d_mask.p, edge_mask, (size_t)e->E, cudaMemcpyHostToDevice, e->stream));
    e->last_kernel = "cert_expm_kernel + cert_inside_kernel + cert_outside_kernel";
    return cert_outside_query(e, CERT_DERIV, edge_mask, site_lo, site_hi, sum_lo, sum_hi);
}

extern "C" int plf_edge_expect_certified(plf_engine *e, double delta_rate, double delta_q, int kind, const double *l_hi,
                                         const double *l_lo, const unsigned char *edge_mask, double *site_lo, double *site_hi,
                                         double *sum_lo, double *sum_hi)
{
    if (!e) return -1;
    if (cert_check(e, "plf_edge_expect_certified", delta_rate, delta_q)) return -1;
    if (kind != PLF_KIND_DWELL && kind != PLF_KIND_TRANS) FAIL(e, "plf_edge_expect_certified: invalid kind %d", kind);
    if (!l_hi) FAIL(e, "plf_edge_expect_certified: l_hi is required");
    CK(e, cudaSetDevice(e->device));
    if (resolve_pending(e)) return -1;
    const int n = e->n, C = e->C, E = e->E;
    if (E == 0) return 0;
    const size_t nn = (size_t)n * n;
    ENSURE(e, e->c_ws, sizeof(double) * C * E * 18 * nn + 8);
    ENSURE(e, e->c_Dlo, sizeof(double) * C * E * nn + 8);
    ENSURE(e, e->c_Dhi, sizeof(double) * C * E * nn + 8);
    if (cert_prepare(e, delta_rate, delta_q, false)) return -1;
    ENSURE(e, e->d_mask, (size_t)E);
    if (edge_mask) CK(e, cudaMemcpyAsync(e->d_mask.p, edge_mask, (size_t)E, cudaMemcpyHostToDevice, e->stream));
    if (upload_L(e, l_hi, l_lo)) return -1;
    cert_frechet_kernel<<<dim3(E, C), 128, 0, e->stream>>>(n, E, C, e->d_qhi.as<double>(), e->d_qlo.as<double>(), e->d_edge_rates.as<double>(),
                                                           e->d_cat_rates.as<double>(), delta_rate, delta_q, e->d_lhi.as<double>(),
                                                           l_lo ? e->d_llo.as<double>() : nullptr, kind == PLF_KIND_TRANS,
                                                           edge_mask ? e->d_mask.as<unsigned char>() : nullptr, e->c_ws.as<double>(),
                                                           e->c_Dlo.as<double>(), e->c_Dhi.as<double>());
    KCHECK(e);
    e->last_kernel = "cert_expm_kernel + cert_frechet_kernel + cert_inside_kernel + cert_outside_kernel";
    return cert_outside_query(e, CERT_EXPECT, edge_mask, site_lo, site_hi, sum_lo, sum_hi);
}

extern "C" int plf_marginal_certified(plf_engine *e, double delta_rate, double delta_q, double *site_lo, double *site_hi,
                                      double *sum_lo, double *sum_hi)
{
    if (!e) return -1;
    if (cert_check(e, "plf_marginal_certified", delta_rate, delta_q)) return -1;
    CK(e, cudaSetDevice(e->device));
    if (resolve_pending(e)) return -1;
    if (cert_prepare(e, delta_rate, delta_q, false)) return -1;
    e->last_kernel = "cert_expm_kernel + cert_inside_kernel + cert_outside_kernel";
    return cert_outside_query(e, CERT_MARGINAL, nullptr, site_lo, site_hi, sum_lo, sum_hi);
}

/* ------------------------------------------------------------------ */
/* site-pattern compression                                            */
/* ------------------------------------------------------------------ */

extern "C" int plf_compress_patterns(plf_engine *e, int64_t S, int N, const void *codes, int code_bytes,
                                     int64_t *n_patterns, void *codes_out, int64_t *counts_out, int64_t *site_to_pattern)
{
    if (!e) return -1;
    if (S < 0 || N <= 0 || !codes || !n_patterns) FAIL(e, "plf_compress_patterns: bad arguments");
    if (code_bytes != 1 && code_bytes != 4) FAIL(e, "plf_compress_patterns: code_bytes must be 1 or 4");
    if (S >= ((int64_t)1 << 31) - 1) FAIL(e, "plf_compress_patterns: more than 2^31 - 2 sites");
    *n_patterns = 0;
    if (S == 0) return 0;
    CK(e, cudaSetDevice(e->device));
    const int row_bytes = N * code_bytes;
    size_t M = 1;
    while (M < (size_t)S * 2) M <<= 1;
    DevBuf d_in, d_table, d_first, d_slot, d_flags, d_scan, d_bsum, d_map, d_counts, d_out, d_total;
    const int nblocks = (int)((S + 1023) / 1024);
    ENSURE(e, d_in, (size_t)S * row_bytes);
    ENSURE(e, d_table, sizeof(int) * M);
    ENSURE(e, d_first, sizeof(int) * M);
    ENSURE(e, d_slot, sizeof(int) * S);
    ENSURE(e, d_flags, sizeof(int) * S);
    ENSURE(e, d_scan, sizeof(int) * S);
    ENSURE(e, d_bsum, sizeof(int) * (nblocks + 1));
    ENSURE(e, d_map, sizeof(int) * S);
    ENSURE(e, d_counts, sizeof(int) * S);
    ENSURE(e, d_out, (size_t)S * row_bytes);
    ENSURE(e, d_total, sizeof(int));
    CK(e, cudaMemcpyAsync(d_in.p, codes, (size_t)S * row_bytes, cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaMemsetAsync(d_table.p, 0xFF, sizeof(int) * M, e->stream));          /* PC_EMPTY */
    CK(e, cudaMemsetAsync(d_first.p, 0x7F, sizeof(int) * M, e->stream));          /* large */
    CK(e, cudaMemsetAsync(d_counts.p, 0, sizeof(int) * S, e->stream));
    const unsigned gs = (unsigned)((S + 255) / 256);
    pc_insert_kernel<<<gs, 256, 0, e->stream>>>(d_in.as<unsigned char>(), S, row_bytes, d_table.as<int>(), (unsigned long long)(M - 1), d_slot.as<int>());
    KCHECK(e);
    pc_first_kernel<<<gs, 256, 0, e->stream>>>(S, d_slot.as<int>(), d_first.as<int>());
    KCHECK(e);
    pc_flag_kernel<<<gs, 256, 0, e->stream>>>(S, d_slot.as<int>(), d_first.as<int>(), d_flags.as<int>());
    KCHECK(e);
    pc_block_sum_kernel<<<nblocks, 1024, 0, e->stream>>>(d_flags.as<int>(), S, d_bsum.as<int>());
    KCHECK(e);
    pc_scan_sums_kernel<<<1, 1024, 0, e->stream>>>(d_bsum.as<int>(), nblocks, d_total.as<int>());
    KCHECK(e);
    pc_scan_final_kernel<<<nblocks, 1024, 0, e->stream>>>(d_flags.as<int>(), S, d_bsum.as<int>(), d_scan.as<int>());
    KCHECK(e);
    pc_emit_kernel<<<gs, 256, 0, e->stream>>>(d_in.as<unsigned char>(), S, row_bytes, d_slot.as<int>(), d_first.as<int>(), d_scan.as<int>(),
                                              d_flags.as<int>(), d_map.as<int>(), d_counts.as<int>(), d_out.as<unsigned char>());
    KCHECK(e);
    int total = 0;
    CK(e, cudaMemcpyAsync(&total, d_total.p, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    *n_patterns = total;
    if (codes_out) CK(e, cudaMemcpyAsync(codes_out, d_out.p, (size_t)total * row_bytes, cudaMemcpyDeviceToHost, e->stream));
    std::vector<int> tmp;
    if (counts_out) {
        tmp.resize(total);
        CK(e, cudaMemcpyAsync(tmp.data(), d_counts.p, sizeof(int) * total, cudaMemcpyDeviceToHost, e->stream));
        CK(e, cudaStreamSynchronize(e->stream));
        for (int i = 0; i < total; i++) counts_out[i] = tmp[i];
    }
    if (site_to_pattern) {
        tmp.resize(S);
        CK(e, cudaMemcpyAsync(tmp.data(), d_map.p, sizeof(int) * S, cudaMemcpyDeviceToHost, e->stream));
        CK(e, cudaStreamSynchronize(e->stream));
        for (int64_t i = 0; i < S; i++) site_to_pattern[i] = tmp[i];
    }
    CK(e, cudaStreamSynchronize(e->stream));
    return 0;
}

/* ------------------------------------------------------------------ */
/* multi-GPU                                                           */
/* ------------------------------------------------------------------ */

extern "C" int plf_comm_unique_id(char id[128])
{
    if (!g_nccl.load()) { fprintf(stderr, "plf_comm_unique_id: cannot load libnccl.so.2\n"); return -1; }
    plf_nccl_id u;
    if (g_nccl.GetUniqueId(&u) != 0) return -1;
    memcpy(id, u.internal, 128);
    return 0;
}

extern "C" int plf_comm_pause(plf_engine *e, int paused)
{
    if (!e) return -1;
    e->comm_paused = paused != 0;
    return 0;
}

extern "C" int plf_comm_init(plf_engine *e, int nranks, int rank, const char id[128])
{
    if (!e) return -1;
    if (!g_nccl.load()) FAIL(e, "cannot load libnccl.so.2: %s", dlerror());
    CK(e, cudaSetDevice(e->device));
    plf_nccl_id u;
    memcpy(u.internal, id, 128);
    int r = g_nccl.CommInitRank(&e->comm, nranks, u, rank);
    if (r != 0) { e->comm = nullptr; FAIL(e, "ncclCommInitRank failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?"); }
    e->nranks = nranks;
    e->rank = rank;
    /* Peer-memory path for the short sum vectors: every rank exports an inbox through CUDA IPC, the handles travel once
     * through ncclAllGather, and from then on the all-reduce is one small kernel of P2P stores and loads
     * (peer_allreduce_kernel).  Any failure here simply leaves the NCCL path in place. */
    e->peer_ready = false;
    if (nranks <= PLF_PEER_MAX && g_nccl.AllGather && !getenv("PLF_NO_PEER_ALLREDUCE")) {
        const size_t bytes = sizeof(double) * (size_t)PLF_PEER_MAX * 2 * PLF_PEER_CAP + sizeof(unsigned long long) * PLF_PEER_MAX * 2;
        bool ok = cudaMalloc(&e->peer_local, bytes) == cudaSuccess && cudaMemset(e->peer_local, 0, bytes) == cudaSuccess;
        cudaIpcMemHandle_t mine;
        char *d_h = nullptr;
        std::vector<cudaIpcMemHandle_t> all(nranks);
        ok = ok && cudaIpcGetMemHandle(&mine, e->peer_local) == cudaSuccess;
        ok = ok && cudaMalloc((void **)&d_h, sizeof(mine) * (nranks + 1)) == cudaSuccess;
        /* the collective below must be entered by every rank, whatever happened locally: a failed rank sends zeros */
        if (!ok) memset(&mine, 0, sizeof(mine));
        if (d_h) {
            cudaMemcpyAsync(d_h + sizeof(mine) * nranks, &mine, sizeof(mine), cudaMemcpyHostToDevice, e->stream);
            const int rr = g_nccl.AllGather(d_h + sizeof(mine) * nranks, d_h, sizeof(mine), /*ncclChar*/ 0, e->comm, e->stream);
            ok = ok && rr == 0;
            cudaMemcpyAsync(all.data(), d_h, sizeof(mine) * nranks, cudaMemcpyDeviceToHost, e->stream);
            ok = (cudaStreamSynchronize(e->stream) == cudaSuccess) && ok;
            cudaFree(d_h);
        }
        const cudaIpcMemHandle_t zero = {};
        for (int p = 0; ok && p < nranks; p++) if (!memcmp(&all[p], &zero, sizeof(zero))) ok = false;       /* some rank could not export */
        for (int p = 0; ok && p < nranks; p++) {
            if (p == rank) { e->peer_ptr[p] = e->peer_local; continue; }
            if (cudaIpcOpenMemHandle(&e->peer_ptr[p], all[p], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { ok = false; cudaGetLastError(); }
        }
        if (ok && !e->d_peer_ptrs.ensure(sizeof(void *) * PLF_PEER_MAX))
            ok = cudaMemcpy(e->d_peer_ptrs.p, e->peer_ptr, sizeof(void *) * PLF_PEER_MAX, cudaMemcpyHostToDevice) == cudaSuccess;
        else ok = false;
        /* every rank takes the peer path or none does */
        double *d_ok = nullptr;
        double h_ok = ok ? 1.0 : 0.0;
        if (cudaMalloc((void **)&d_ok, sizeof(double)) == cudaSuccess) {
            cudaMemcpyAsync(d_ok, &h_ok, sizeof(double), cudaMemcpyHostToDevice, e->stream);
            const int rr = g_nccl.AllReduce(d_ok, d_ok, 1, /*ncclDouble*/ 8, /*ncclSum*/ 0, e->comm, e->stream);
            cudaMemcpyAsync(&h_ok, d_ok, sizeof(double), cudaMemcpyDeviceToHost, e->stream);
            if (cudaStreamSynchronize(e->stream) != cudaSuccess || rr != 0) h_ok = 0.0;
            cudaFree(d_ok);
        } else {
            FAIL(e, "plf_comm_init: out of device memory");
        }
        e->peer_ready = (h_ok == (double)nranks);
        e->peer_seq = 0;
        cudaGetLastError();
    }
    return 0;
}
