// unc_abi.cu -- kernels + C-ABI (include/unc_b200.h) of the B200-native `uncalled map` path.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -fmad=false --shared
// This translation unit contains NO CPU implementation of the path: every compute entry
// point launches the sm_100a kernels below or fails with a CUDA status.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <mutex>
#include <string>
#include <vector>

#include "unc_device.cuh"
#include "unc_k1.cuh"
#include "unc_stream.cuh"
#include "../../include/unc_b200.h"
#include "unc_host_index.hpp"
#include "unc_host_params.hpp"
#include "unc_ordered_logic.hpp"

static_assert(sizeof(DevRec) == sizeof(unc_paf_rec), "DevRec must mirror unc_paf_rec");
static_assert(sizeof(DevReadDesc) == 32, "DevReadDesc layout");

// ------------------------------------------------------------------ kernels

#ifndef K2_WARPS
#define K2_WARPS 14         /* 1 tracker warp + (K2_WARPS-1) worker warps per read */
#endif
#ifndef K2_MIN_CTAS
#define K2_MIN_CTAS 2       /* second worker structure: 2 CTAs x 14 warps per SM (72 registers) measured best */
#endif
#define K2_MIN_CTAS_V1 (K2_WARPS > 8 ? 1 : 2)    /* first structure (exact-ties kernels): 127 registers */
#define K2_THREADS (K2_WARPS * 32)
static_assert(K2_WARPS >= 2 && K2_WARPS - 1 <= K2_MAXSEG, "worker warps must fit the sort segments");

__global__ void k_kmer_ranges(DevIndex ix, uint2 *out) {
    u32 k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < UNC_NKMER) out[k] = unc_kmer_range_compute(ix, k);
}

// the GPU-side Occ layout (unc_k2v2.cuh): one 32-byte block per 64 BWT positions
__global__ void k_occ2_build(const uint4 *bwt, uint4 *out, u32 n_blk) {
    u32 j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n_blk) unc_occ2_build_block(bwt, j, out);
}

// bwt_sa(k) for every row: turns the mapper's <=31-step LF walk per seed into one load.
__global__ void k_sa_expand(DevIndex ix, u32 *out, u32 n_rows) {
    u32 k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_rows) return;
    u32 a = 0, b = 0;
    out[k] = unc_sa(ix, k, &a, &b);
}

// K1: warp-per-read event detection (unc_k1.cuh).  K1_WARPS independent warps per CTA, each
// with its own shared-memory tile buffers and mbarrier; reads are pulled from an atomic queue.
#ifndef K1_WARPS
#define K1_WARPS 4
#endif
#ifndef K1_MIN_CTAS
#define K1_MIN_CTAS 1
#endif
__global__ void __launch_bounds__(K1_WARPS * 32, K1_MIN_CTAS) k1_events(DevBatch B, DevParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    K1WarpSmem *sm = (K1WarpSmem *) smem_raw + (threadIdx.x >> 5);
    unc_k1_warp_main(B, p, sm);
}
// reads whose samples fail the exactness condition of the warp-parallel sums: serial routine
__global__ void __launch_bounds__(128) k1_fallback(DevBatch B, DevParams p) {
    u32 r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < B.n_reads && B.k1_flags[r]) unc_k1_read(B, p, r);
}
// normaliser statistics (sequential double reductions), one thread per read
__global__ void __launch_bounds__(128) k1_norm(DevBatch B, DevParams p) {
    u32 r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < B.n_reads && !B.k1_flags[r]) unc_k1_norm_read(B, p, r);
}

// Persistent CTA-per-read mapper.  Each CTA stages the pore model, the 1024 k-mer FM ranges
// and the thresholds in shared memory, then pulls reads from a global queue; the K2_WARPS warps
// of the CTA cooperate on every event of the read (chained scans through shared memory).
#define K2_MAP_KERNEL(NAME, EXACT, FLAGS)                                                                                       \
    __global__ void __launch_bounds__(K2_THREADS, (EXACT) ? K2_MIN_CTAS_V1 : K2_MIN_CTAS)                                  \
    NAME(DevIndex ix, DevParams p, DevBatch B, DevWork W0, DevWorkStrides S) {                                             \
        extern __shared__ __align__(16) unsigned char smem_raw[];                                                          \
        unc_k2_cta_main<EXACT, FLAGS>(ix, p, B, unc_work_slot(W0, S, blockIdx.x), (K2Shared *) smem_raw);                 \
    }
K2_MAP_KERNEL(k2_map, false, false)
// ordered mode (unc_map_batch_ordered): per-read sources_added_ words in and out (kept out of k2_map, whose code is
// the build that was measured)
K2_MAP_KERNEL(k2_map_ord, false, true)
// the exact-ties kernel (unc_pool_set_tie_order): the same mapper with the reference's unstable child sort run serially
K2_MAP_KERNEL(k2_map_exact, true, true)

// ordered mode: per read the 1024-bit mask of the k-mers that pass the first event's fresh-source tests
// (block = read, thread = k-mer; word k>>5, bit k&31 = the ballot of warp k>>5)
__global__ void __launch_bounds__(UNC_NKMER) k_event0_cands(DevIndex ix, DevParams p, DevBatch B, u32 *cand) {
    const u32 r = blockIdx.x, k = threadIdx.x;
    const u32 m = __ballot_sync(0xFFFFFFFFu, unc_event0_cand(ix, p, B, r, k));
    if ((k & 31u) == 0) cand[(size_t) r * 32 + (k >> 5)] = m;
}

__global__ void k_match_probs(DevIndex ix, float event, float *out) {
    u32 k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < UNC_NKMER) out[k] = unc_match_prob(event, ix.lv_mean[k], ix.lv_var2[k], ix.lognorm[k]);
}

__global__ void k_fm_neighbors(DevIndex ix, u32 n, const u64 *st, const u64 *en, const u8 *base, u64 *ost, u64 *oen) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u32 ns[4], ne[4], nb = 0, c = base[i];
    u32 ok = unc_neighbors(ix, (u32) st[i], (u32) en[i], 1u << c, ns, ne, &nb);
    if (!((ok >> c) & 1u)) {   // empty range: report it the way get_neighbor does (start = end + 1 ...)
        ns[c] = unc_L2(ix, c) + unc_occ(ix, (u32) st[i] - 1u, c, &nb) + 1u;
        ne[c] = unc_L2(ix, c) + unc_occ(ix, (u32) en[i], c, &nb);
    }
    ost[i] = ns[c];
    oen[i] = ne[c];
}

__global__ void k_fm_sa(DevIndex ix, u32 n, const u64 *rows, u64 *out) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u32 a = 0, b = 0;
    // widen like the reference: sa[0] = (u64)-1
    u32 v = unc_sa(ix, (u32) rows[i], &a, &b);
    out[i] = v;
}

// ------------------------------------------------------------------ host state

static thread_local std::string g_err;
static int g_device = 0;

// cudaFuncAttributeMaxDynamicSharedMemorySize is per function and process-wide (per device): pools with different
// max_paths need different amounts, so the attribute is only ever RAISED (a running maximum per kernel and device).
template <typename F>
static cudaError_t raise_dyn_smem(F kernel, size_t bytes) {
    static std::mutex mu;
    static std::vector<std::pair<std::pair<const void *, int>, size_t>> seen;
    std::lock_guard<std::mutex> lk(mu);
    int dev = 0;
    cudaGetDevice(&dev);
    const std::pair<const void *, int> key((const void *) kernel, dev);
    for (auto &e : seen)
        if (e.first == key) {
            if (e.second >= bytes) return cudaSuccess;
            cudaError_t r = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
            if (r == cudaSuccess) e.second = bytes;
            return r;
        }
    cudaError_t r = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    if (r == cudaSuccess) seen.push_back({key, bytes});
    return r;
}

static int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}
#define CUDA_TRY(x)                                                                                   \
    do {                                                                                              \
        cudaError_t _e = (x);                                                                         \
        if (_e != cudaSuccess)                                                                        \
            return fail(UNC_E_CUDA, std::string(#x) + ": " + cudaGetErrorString(_e));                  \
    } while (0)

struct unc_index {
    HostIndex h;
    DevIndex ix;
    int device = 0;
    std::vector<uint2> kmer_range;  // host copy
    void *d_bwt = nullptr, *d_sa = nullptr, *d_kr = nullptr, *d_model = nullptr, *d_thresh = nullptr;
    void *d_seq_off = nullptr, *d_seq_len = nullptr, *d_sa_full = nullptr, *d_occ2 = nullptr, *d_krank = nullptr;
    size_t device_bytes = 0;
};

struct unc_pool {
    const unc_index *idx = nullptr;
    unc_params prm;
    DevParams dp;
    uint32_t max_reads = 0;
    uint64_t max_samples = 0;
    uint32_t ev_stride = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // [5]: end of k1_events
    // batch buffers
    void *d_samples = nullptr;
    DevReadDesc *d_reads = nullptr, *h_reads = nullptr;
    float *d_events = nullptr, *d_normed = nullptr, *d_scale = nullptr, *d_shift = nullptr, *d_mel = nullptr;
    u32 *d_n_events = nullptr, *d_queue = nullptr, *d_k1_flags = nullptr;   // d_queue: [k2 queue, k1 queue, 4 x k1 stats]
    uint32_t k1_grid = 0;
    DevRec *d_out = nullptr;
    unsigned long long *d_dbg = nullptr;
    unc_paf_rec *h_out = nullptr;  // pinned staging
    // workspaces
    DevWork W;
    DevWorkStrides strides{};
    uint32_t n_slots = 0, grid = 0;
    size_t smem = 0;
    unc_timing last;
    cudaEvent_t ev_user[2] = {nullptr, nullptr};   // unc_pool_record / unc_pool_elapsed
    uint32_t pending_n = 0;      // reads of a submitted, not yet collected batch (unc_map_batch_submit / _wait)
    uint64_t pending_h2d = 0;
    // ordered mode (unc_map_batch_ordered): per-read sources_added_ words in / out, allocated on first use
    int tie_order = 0;           // unc_pool_set_tie_order: 0 = emission order (k2_map), 1 = the reference's pdqsort (k2_map_exact)
    u32 *d_flags_in = nullptr, *d_flags_out = nullptr, *d_cand = nullptr;
    bool want_cand = false;      // the next batch_enqueue also launches k_event0_cands
};

extern "C" {

const char *unc_strerror(int s) {
    switch (s) {
        case UNC_OK: return "ok";
        case UNC_E_ARG: return "bad argument";
        case UNC_E_IO: return "index I/O error";
        case UNC_E_CUDA: return "CUDA error";
        case UNC_E_NO_DEVICE: return "no CUDA device";
        case UNC_E_TOO_LARGE: return "index or batch too large for the device image";
        case UNC_E_NOMEM: return "out of memory";
        case UNC_E_OVERFLOW: return "per-read device workspace overflow";
    }
    return "unknown status";
}

const char *unc_last_error(void) { return g_err.c_str(); }

int unc_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int unc_init(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) return fail(UNC_E_NO_DEVICE, "no CUDA device (the product has no CPU fallback)");
    if (device < 0 || device >= n) return fail(UNC_E_ARG, "device out of range");
    CUDA_TRY(cudaSetDevice(device));
    g_device = device;
    return UNC_OK;
}

int unc_shutdown(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) == cudaSuccess && g_device < n && cudaSetDevice(g_device) == cudaSuccess) {
        unc_dtw_release();
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) return fail(UNC_E_CUDA, std::string("cudaDeviceSynchronize: ") + cudaGetErrorString(e));
    }
    g_device = 0;
    g_err.clear();
    return UNC_OK;
}

int unc_params_default(unc_params *p) {
    if (!p) return fail(UNC_E_ARG, "null params");
    unc_fill_default_params(p);
    return UNC_OK;
}

static int upload(void **dst, const void *src, size_t bytes, size_t pad, size_t *total) {
    CUDA_TRY(cudaMalloc(dst, bytes + pad));
    if (pad) CUDA_TRY(cudaMemset((char *) *dst + bytes, 0, pad));
    CUDA_TRY(cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice));
    *total += bytes + pad;
    return UNC_OK;
}

int unc_index_load(const char *bwa_prefix, const char *preset, const char *model_table_path, unc_index **out) {
    if (!bwa_prefix || !out || !model_table_path) return fail(UNC_E_ARG, "null argument");
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0)
        return fail(UNC_E_NO_DEVICE, "no CUDA device (the product has no CPU fallback)");
    CUDA_TRY(cudaSetDevice(g_device));
    unc_index *x = new unc_index();
    x->device = g_device;
    if (!hix_load_model(x->h, model_table_path) || !hix_load(x->h, bwa_prefix, preset ? preset : "default")) {
        std::string e = x->h.error;
        delete x;
        return fail(UNC_E_IO, e);
    }
    HostIndex &h = x->h;
    if (h.seq_len >= 0xFFFFFF00ull) {
        delete x;
        return fail(UNC_E_TOO_LARGE, "FM index longer than 2^32 rows is not supported by the u32 device image");
    }
    int rc;
#define UP(dst, src, bytes, pad) if ((rc = upload(&(dst), (src), (bytes), (pad), &x->device_bytes)) != UNC_OK) { unc_index_free(x); return rc; }
    UP(x->d_bwt, h.bwt.data(), h.bwt.size() * 4, 64);
    UP(x->d_sa, h.sa32.data(), h.sa32.size() * 4, 16);
    std::vector<float> model(3 * 1024);
    std::copy(h.lv_mean.begin(), h.lv_mean.end(), model.begin());
    std::copy(h.lv_var2.begin(), h.lv_var2.end(), model.begin() + 1024);
    std::copy(h.lognorm.begin(), h.lognorm.end(), model.begin() + 2048);
    UP(x->d_model, model.data(), model.size() * 4, 0);
    UP(x->d_thresh, h.thresh, 64 * 4, 0);
    std::vector<u64> so(h.offsets.begin(), h.offsets.end());
    if (so.empty()) so.push_back(0);
    std::vector<u32> sl(h.lens.begin(), h.lens.end());
    if (sl.empty()) sl.push_back(0);
    UP(x->d_seq_off, so.data(), so.size() * 8, 0);
    UP(x->d_seq_len, sl.data(), sl.size() * 4, 0);
#undef UP
    if (cudaMalloc(&x->d_kr, 1024 * sizeof(uint2)) != cudaSuccess) { unc_index_free(x); return fail(UNC_E_CUDA, "cudaMalloc kmer ranges"); }
    x->device_bytes += 1024 * sizeof(uint2);
    DevIndex &ix = x->ix;
    ix.bwt = (const uint4 *) x->d_bwt;
    ix.sa = (const u32 *) x->d_sa;
    ix.kmer_range = (const uint2 *) x->d_kr;
    ix.lv_mean = (const float *) x->d_model;
    ix.lv_var2 = ix.lv_mean + 1024;
    ix.lognorm = ix.lv_mean + 2048;
    ix.thresh = (const float *) x->d_thresh;
    ix.primary = (u32) h.primary;
    ix.seq_len = (u32) h.seq_len;
    for (int i = 0; i < 5; i++) ix.L2[i] = (u32) h.L2[i];
    ix.start_bits = 64 - __builtin_clzll(h.seq_len ? h.seq_len : 1);
    ix.sa_full = nullptr;
    ix.occ2 = nullptr; ix.kt = nullptr;
    {   // expanded suffix array (4 bytes per FM row); skipped when device memory is short
        size_t free_b = 0, total_b = 0;
        const size_t need = ((size_t) h.seq_len + 1) * 4;
        if (!getenv("UNC_NO_SA_EXPAND") && cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && need < free_b / 4 &&
            cudaMalloc(&x->d_sa_full, need) == cudaSuccess) {
            u32 n_rows = (u32) h.seq_len + 1u;
            k_sa_expand<<<(n_rows + 255) / 256, 256>>>(ix, (u32 *) x->d_sa_full, n_rows);
            if (cudaDeviceSynchronize() == cudaSuccess) { ix.sa_full = (const u32 *) x->d_sa_full; x->device_bytes += need; }
            else { unc_index_free(x); return fail(UNC_E_CUDA, "k_sa_expand failed"); }
        }
    }
    k_kmer_ranges<<<4, 256>>>(ix, (uint2 *) x->d_kr);
    x->kmer_range.resize(1024);
    cudaError_t e = cudaMemcpy(x->kmer_range.data(), x->d_kr, 1024 * sizeof(uint2), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) { unc_index_free(x); return fail(UNC_E_CUDA, std::string("k_kmer_ranges: ") + cudaGetErrorString(e)); }
    {   // GPU-side layouts of the mapper's second structure: 32-byte Occ blocks, k-mer rank tables
        const u32 n_blk = (u32) (h.bwt.size() / 16) * 2u;
        if (cudaMalloc(&x->d_occ2, (size_t) n_blk * 32 + 64) != cudaSuccess) { unc_index_free(x); return fail(UNC_E_CUDA, "cudaMalloc occ2"); }
        cudaMemset((char *) x->d_occ2 + (size_t) n_blk * 32, 0, 64);
        k_occ2_build<<<(n_blk + 255) / 256, 256>>>(ix.bwt, (uint4 *) x->d_occ2, n_blk);
        K2V2Tab kt;
        if (!hix_k2v2_tab(x->kmer_range.data(), kt)) { unc_index_free(x); return fail(UNC_E_TOO_LARGE, "more overlapping k-mer FM ranges than the bucket table holds"); }
        if (cudaMalloc(&x->d_krank, sizeof(kt)) != cudaSuccess ||
            cudaMemcpy(x->d_krank, &kt, sizeof(kt), cudaMemcpyHostToDevice) != cudaSuccess ||
            cudaDeviceSynchronize() != cudaSuccess) { unc_index_free(x); return fail(UNC_E_CUDA, "occ2 / k-mer bucket tables"); }
        ix.occ2 = (const uint4 *) x->d_occ2;
        ix.kt = (const K2V2Tab *) x->d_krank;
        x->device_bytes += (size_t) n_blk * 32 + 64 + sizeof(kt);
    }
    *out = x;
    return UNC_OK;
}

int unc_index_get_info(const unc_index *x, unc_index_info *info) {
    if (!x || !info) return fail(UNC_E_ARG, "null argument");
    info->n_rows = x->h.seq_len;
    info->n_seqs = (int32_t) x->h.names.size();
    info->device = x->device;
    info->device_bytes = x->device_bytes;
    info->n_kmer_groups = 1024;
    return UNC_OK;
}

int unc_index_seq(const unc_index *x, int rid, const char **name, uint64_t *len) {
    if (!x || rid < 0 || rid >= (int) x->h.names.size()) return fail(UNC_E_ARG, "rid out of range");
    if (name) *name = x->h.names[rid].c_str();
    if (len) *len = x->h.lens[rid];
    return UNC_OK;
}

int unc_index_kmer_range(const unc_index *x, uint32_t kmer, uint64_t *start, uint64_t *end) {
    if (!x || kmer >= 1024) return fail(UNC_E_ARG, "bad kmer");
    *start = x->kmer_range[kmer].x;
    *end = x->kmer_range[kmer].y;
    return UNC_OK;
}

int unc_index_thresholds(const unc_index *x, float out[64]) {
    if (!x || !out) return fail(UNC_E_ARG, "null argument");
    memcpy(out, x->h.thresh, 64 * sizeof(float));
    return UNC_OK;
}

void unc_index_free(unc_index *x) {
    if (!x) return;
    cudaFree(x->d_bwt); cudaFree(x->d_sa); cudaFree(x->d_kr); cudaFree(x->d_model); cudaFree(x->d_thresh);
    cudaFree(x->d_seq_off); cudaFree(x->d_seq_len); cudaFree(x->d_sa_full); cudaFree(x->d_occ2); cudaFree(x->d_krank);
    delete x;
}

int unc_pool_create(const unc_index *idx, const unc_params *prm, uint32_t max_reads, uint64_t max_samples,
                    unc_pool **out) {
    if (!idx || !prm || !out || max_reads == 0 || max_samples == 0) return fail(UNC_E_ARG, "null/zero argument");
    std::string err;
    if (unc_check_params(*prm, err)) return fail(UNC_E_ARG, err);
    CUDA_TRY(cudaSetDevice(idx->device));
    unc_pool *P = new unc_pool();
    P->idx = idx;
    P->prm = *prm;
    P->dp = unc_make_dev_params(*prm, idx->h);
    P->max_reads = max_reads;
    P->max_samples = max_samples;
    memset(&P->last, 0, sizeof(P->last));
    int rc = UNC_OK;
    auto bail = [&](int code, const std::string &m) { unc_pool_free(P); return fail(code, m); };
#define PT(x) do { cudaError_t _e = (x); if (_e != cudaSuccess) return bail(UNC_E_CUDA, std::string(#x) + ": " + cudaGetErrorString(_e)); } while (0)
    PT(cudaStreamCreateWithFlags(&P->stream, cudaStreamNonBlocking));
    for (int i = 0; i < 6; i++) PT(cudaEventCreate(&P->ev[i]));
    cudaDeviceProp prop;
    PT(cudaGetDeviceProperties(&prop, idx->device));
    P->smem = K2_SMEM_BYTES(prm->max_paths);
    PT(raise_dyn_smem(k2_map, P->smem));
    int per_sm = 0;
    PT(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k2_map, K2_THREADS, P->smem));
    if (per_sm < 1) return bail(UNC_E_CUDA, "k2_map does not fit on an SM");
    if (const char *e = getenv("UNC_K2_CTAS_PER_SM")) { int v = atoi(e); if (v >= 1 && v < per_sm) per_sm = v; }   // tuning knob
    uint32_t grid = (uint32_t) prop.multiProcessorCount * (uint32_t) per_sm;
    if (grid > max_reads) grid = max_reads;
    {
        const size_t k1_smem = (size_t) K1_WARPS * sizeof(K1WarpSmem);
        PT(raise_dyn_smem(k1_events, k1_smem));
        int k1_per_sm = 0;
        PT(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&k1_per_sm, k1_events, K1_WARPS * 32, k1_smem));
        if (k1_per_sm < 1) return bail(UNC_E_CUDA, "k1_events does not fit on an SM");
        P->k1_grid = (uint32_t) prop.multiProcessorCount * (uint32_t) k1_per_sm;
    }
    // per-slot workspace sizes
    const size_t maxp = prm->max_paths;
    const size_t nchmax = (maxp + 31) / 32;
    DevWorkStrides &S = P->strides;
    S.paths = 2 * (nchmax * 160 + maxp) * 2;   // uint4: chunk-local child slots + sources, two generations
    S.hist = 24 * (nchmax * 160 + maxp);      // uint2: (C, parent) per record index, 24 generations
    S.ckey = 2 * maxp;        // uint4
    S.cks = nchmax * 160;     // uint4
    S.elist = nchmax * 32;    // uint4
    S.order = 2 * maxp;       // u32
    uint64_t longest = max_samples < 0xFFFFFFFFull ? max_samples : 0xFFFFFFFFull;
    // seed clusters: at most a few per event in practice; blocks are >= half full after splits
    uint64_t ev_cap = std::min<uint64_t>(prm->max_events, longest / 3 + 16);
    uint64_t mb = std::max<uint64_t>(1024, ev_cap * 2);
    mb = std::min<uint64_t>(mb, 1u << 17);
    const size_t rl_cap = 64 * 1024;   // seed rows of one event (typically tens)
    S.rlist = 2 * rl_cap;
    S.clu = (size_t) mb * UNC_BLK * 2;
    S.dir = (size_t) mb + 1;
    P->W.rl_cap = (u32) rl_cap;
    P->W.max_blocks = (u32) mb;
    size_t per_slot = (S.paths + S.ckey + 2 * S.cks + S.elist) * 16 + S.hist * 8 + S.order * 4 + S.rlist * 8 + S.clu * 16 + S.dir * 16;
    size_t free_b = 0, total_b = 0;
    PT(cudaMemGetInfo(&free_b, &total_b));
    size_t fixed = max_samples * 4 + (size_t) max_reads * (sizeof(DevReadDesc) + sizeof(DevRec) + 20) + (64u << 20);
    P->ev_stride = 0;
    if (free_b < fixed + per_slot) return bail(UNC_E_NOMEM, "not enough device memory for the pool");
    size_t budget = (size_t) ((free_b - fixed) * 0.85);
    while ((size_t) grid * per_slot > budget && grid > 1) grid--;
    P->grid = grid;
    P->n_slots = grid;
    PT(cudaMalloc(&P->W.paths, (size_t) P->n_slots * S.paths * 16));
    PT(cudaMalloc(&P->W.ckey, (size_t) P->n_slots * S.ckey * 16));
    PT(cudaMalloc(&P->W.hist, (size_t) P->n_slots * S.hist * 8));
    PT(cudaMemset(P->W.hist, 0, (size_t) P->n_slots * S.hist * 8));
    PT(cudaMalloc(&P->W.wlist, (size_t) P->n_slots * S.cks * 16));
    PT(cudaMalloc(&P->W.cks, (size_t) P->n_slots * S.cks * 16));
    PT(cudaMalloc(&P->W.elist, (size_t) P->n_slots * S.elist * 16));
    PT(cudaMalloc(&P->W.order, (size_t) P->n_slots * S.order * 4));
    PT(cudaMalloc(&P->W.rlist, (size_t) P->n_slots * S.rlist * 8));
    PT(cudaMalloc(&P->W.clu, (size_t) P->n_slots * S.clu * 16));
    PT(cudaMalloc(&P->W.dir, (size_t) P->n_slots * S.dir * 16));
    PT(cudaMalloc(&P->d_samples, max_samples * 4 + 64));
    PT(cudaMalloc(&P->d_reads, (size_t) max_reads * sizeof(DevReadDesc)));
    PT(cudaMallocHost(&P->h_reads, (size_t) max_reads * sizeof(DevReadDesc)));
    PT(cudaMalloc(&P->d_scale, (size_t) max_reads * 4));
    PT(cudaMalloc(&P->d_shift, (size_t) max_reads * 4));
    PT(cudaMalloc(&P->d_mel, (size_t) max_reads * 4));
    PT(cudaMalloc(&P->d_n_events, (size_t) max_reads * 4));
    PT(cudaMalloc(&P->d_queue, 32));
    PT(cudaMalloc(&P->d_k1_flags, (size_t) max_reads * 4));
    PT(cudaMalloc(&P->d_out, (size_t) max_reads * sizeof(DevRec)));
#ifdef UNC_PHASE_TIMING
    PT(cudaMalloc(&P->d_dbg, (size_t) max_reads * 512 + UNC_PT_TRACE_BYTES));     // counters per read, then the timeline of one read
    PT(cudaMemset(P->d_dbg, 0, (size_t) max_reads * 512 + UNC_PT_TRACE_BYTES));
#endif
    PT(cudaMallocHost(&P->h_out, (size_t) max_reads * sizeof(unc_paf_rec)));
#undef PT
    (void) rc;
    *out = P;
    return UNC_OK;
}

void unc_pool_free(unc_pool *P) {
    if (!P) return;
    cudaFree(P->W.paths); cudaFree(P->W.hist); cudaFree(P->W.wlist); cudaFree(P->W.ckey); cudaFree(P->W.cks); cudaFree(P->W.elist); cudaFree(P->W.order); cudaFree(P->W.rlist); cudaFree(P->W.clu); cudaFree(P->W.dir);
    cudaFree(P->d_samples); cudaFree(P->d_reads); cudaFreeHost(P->h_reads);
    cudaFree(P->d_events); cudaFree(P->d_normed);
    cudaFree(P->d_scale); cudaFree(P->d_shift); cudaFree(P->d_mel); cudaFree(P->d_n_events); cudaFree(P->d_queue); cudaFree(P->d_k1_flags);
    cudaFree(P->d_out); cudaFreeHost(P->h_out); cudaFree(P->d_dbg);
    cudaFree(P->d_flags_in); cudaFree(P->d_flags_out); cudaFree(P->d_cand);
    for (int i = 0; i < 2; i++) if (P->ev_user[i]) cudaEventDestroy(P->ev_user[i]);
    for (int i = 0; i < 6; i++) if (P->ev[i]) cudaEventDestroy(P->ev[i]);
    if (P->stream) cudaStreamDestroy(P->stream);
    delete P;
}

// validates descriptors, stages them, (re)allocates the events buffer; returns the sample span
static int stage_reads(unc_pool *P, const unc_read_desc *reads, uint32_t n, uint64_t *span_bytes, uint32_t *max_n,
                       bool want_normed) {
    if (n == 0 || n > P->max_reads) return fail(UNC_E_ARG, "n_reads outside 1..max_reads");
    uint64_t hi = 0;
    uint32_t mx = 0;
    uint32_t dtype = reads[0].dtype;
    for (uint32_t i = 0; i < n; i++) {
        if (reads[i].dtype != dtype || dtype > 1) return fail(UNC_E_ARG, "mixed or unknown dtype in a batch");
        hi = std::max<uint64_t>(hi, reads[i].offset + reads[i].n_samples);
        mx = std::max(mx, reads[i].n_samples);
        DevReadDesc &d = P->h_reads[i];
        d.offset = reads[i].offset; d.n_samples = reads[i].n_samples; d.dtype = reads[i].dtype;
        d.cal_range = reads[i].cal_range; d.cal_offset = reads[i].cal_offset; d.cal_digit = reads[i].cal_digit;
        d.pad = 0;
    }
    if (hi > P->max_samples) return fail(UNC_E_TOO_LARGE, "batch exceeds the pool's max_samples");
    *span_bytes = hi * (dtype == UNC_DTYPE_F32 ? 4 : 2);
    *max_n = mx;
    uint32_t stride = (mx + 3u) & ~3u;
    if (stride == 0) stride = 4;
    if (stride > P->ev_stride || (want_normed && !P->d_normed)) {
        if (stride > P->ev_stride) {
            cudaFree(P->d_events); P->d_events = nullptr;
            cudaFree(P->d_normed); P->d_normed = nullptr;
            P->ev_stride = stride;
            CUDA_TRY(cudaMalloc(&P->d_events, (size_t) P->max_reads * P->ev_stride * 4));
        }
        if (want_normed && !P->d_normed) CUDA_TRY(cudaMalloc(&P->d_normed, (size_t) P->max_reads * P->ev_stride * 4));
    }
    return UNC_OK;
}

static DevBatch make_batch(unc_pool *P, const void *d_samples, uint64_t samples_bytes, uint32_t n, bool normed) {
    DevBatch B;
    B.samples = d_samples;
    B.samples_bytes = samples_bytes;
    B.k1_queue = P->d_queue + 1;
    B.k1_flags = P->d_k1_flags;
    B.k1_stats = P->d_queue + 2;
    B.reads = P->d_reads;
    B.n_reads = n;
    B.events = P->d_events;
    B.normed = normed ? P->d_normed : nullptr;
    B.ev_stride = P->ev_stride;
    B.n_events = P->d_n_events;
    B.scale = P->d_scale; B.shift = P->d_shift; B.mean_event_len = P->d_mel;
    B.queue = P->d_queue;
    B.dbg = P->d_dbg;
    B.out = P->d_out;
    B.seq_offsets = (const u64 *) P->idx->d_seq_off;
    B.seq_lens = (const u32 *) P->idx->d_seq_len;
    B.n_seqs = (u32) P->idx->h.names.size();
    B.l_pac = (u64) P->idx->h.l_pac;
    return B;
}

// event detection (warp per read) -> serial redo of flagged reads -> normaliser statistics
static void launch_k1(unc_pool *P, const DevBatch &B, uint32_t n, cudaStream_t s) {
    uint32_t g = std::min<uint32_t>(P->k1_grid, (n + K1_WARPS - 1) / K1_WARPS);
    k1_events<<<g, K1_WARPS * 32, (size_t) K1_WARPS * sizeof(K1WarpSmem), s>>>(B, P->dp);
    cudaEventRecord(P->ev[5], s);
    k1_fallback<<<(n + 127) / 128, 128, 0, s>>>(B, P->dp);
    k1_norm<<<(n + 127) / 128, 128, 0, s>>>(B, P->dp);
}

// first half of a batch: everything is put on the pool's stream (copies in, both kernels, copy out), nothing waits
// h_flags_in (ordered mode only): n x 32 sources_added_ words the reads start from; their final words go to d_flags_out.
static int batch_enqueue(unc_pool *P, const unc_read_desc *reads, uint32_t n, const void *samples, bool on_device,
                         const uint32_t *h_flags_in = nullptr) {
    if (!P || !reads || !samples) return fail(UNC_E_ARG, "null argument");
    if (P->pending_n) return fail(UNC_E_ARG, "the pool still holds a submitted batch: call unc_map_batch_wait first");
    CUDA_TRY(cudaSetDevice(P->idx->device));
    uint64_t span = 0;
    uint32_t mx = 0;
    int rc = stage_reads(P, reads, n, &span, &mx, false);
    if (rc) return rc;
    cudaStream_t s = P->stream;
    CUDA_TRY(cudaEventRecord(P->ev[0], s));
    const void *d_samples = samples;
    uint64_t h2d = (uint64_t) n * sizeof(DevReadDesc);
    if (!on_device) {
        CUDA_TRY(cudaMemcpyAsync(P->d_samples, samples, span, cudaMemcpyHostToDevice, s));
        d_samples = P->d_samples;
        h2d += span;
    }
    CUDA_TRY(cudaMemcpyAsync(P->d_reads, P->h_reads, (size_t) n * sizeof(DevReadDesc), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemsetAsync(P->d_queue, 0, 32, s));
    if (P->d_dbg) CUDA_TRY(cudaMemsetAsync(P->d_dbg, 0, (size_t) n * 512, s));      // phase-timing builds only
    CUDA_TRY(cudaEventRecord(P->ev[1], s));
    // the pool's own staging buffer is padded, so whole 16-byte bulk copies may run past `span`
    DevBatch B = make_batch(P, d_samples, on_device ? span : ((span + 15) & ~(uint64_t) 15), n, false);
    if (h_flags_in) {
        if (!P->d_flags_in) {
            CUDA_TRY(cudaMalloc(&P->d_flags_in, (size_t) P->max_reads * 128));
            CUDA_TRY(cudaMalloc(&P->d_flags_out, (size_t) P->max_reads * 128));
            CUDA_TRY(cudaMalloc(&P->d_cand, (size_t) P->max_reads * 128));
            CUDA_TRY(raise_dyn_smem(k2_map_ord, P->smem));
        }
        CUDA_TRY(cudaMemcpyAsync(P->d_flags_in, h_flags_in, (size_t) n * 128, cudaMemcpyHostToDevice, s));
        B.flags_in = P->d_flags_in;
        B.flags_out = P->d_flags_out;
        h2d += (uint64_t) n * 128;
    }
    launch_k1(P, B, n, s);
    if (h_flags_in && P->want_cand) k_event0_cands<<<n, UNC_NKMER, 0, s>>>(P->idx->ix, P->dp, B, P->d_cand);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(P->ev[2], s));
    uint32_t grid = std::min<uint32_t>(P->grid, n);
    if (P->tie_order) k2_map_exact<<<grid, K2_THREADS, P->smem, s>>>(P->idx->ix, P->dp, B, P->W, P->strides);
    else if (h_flags_in) k2_map_ord<<<grid, K2_THREADS, P->smem, s>>>(P->idx->ix, P->dp, B, P->W, P->strides);
    else k2_map<<<grid, K2_THREADS, P->smem, s>>>(P->idx->ix, P->dp, B, P->W, P->strides);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(P->ev[3], s));
    CUDA_TRY(cudaMemcpyAsync(P->h_out, P->d_out, (size_t) n * sizeof(DevRec), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaEventRecord(P->ev[4], s));
    P->pending_n = n;
    P->pending_h2d = h2d;
    return UNC_OK;
}

// second half: wait for the stream, hand the records over, read the event timings
static int batch_finish(unc_pool *P, unc_paf_rec *out) {
    if (!P || !out) return fail(UNC_E_ARG, "null argument");
    if (!P->pending_n) return fail(UNC_E_ARG, "no submitted batch to wait for");
    const uint32_t n = P->pending_n;
    const uint64_t h2d = P->pending_h2d;
    P->pending_n = 0;
    CUDA_TRY(cudaSetDevice(P->idx->device));
    CUDA_TRY(cudaStreamSynchronize(P->stream));
    memcpy(out, P->h_out, (size_t) n * sizeof(unc_paf_rec));
    unc_timing &t = P->last;
    cudaEventElapsedTime(&t.h2d_ms, P->ev[0], P->ev[1]);
    cudaEventElapsedTime(&t.k1_ms, P->ev[1], P->ev[2]);
    cudaEventElapsedTime(&t.k1_events_ms, P->ev[1], P->ev[5]);
    cudaEventElapsedTime(&t.k2_ms, P->ev[2], P->ev[3]);
    cudaEventElapsedTime(&t.d2h_ms, P->ev[3], P->ev[4]);
    cudaEventElapsedTime(&t.total_ms, P->ev[0], P->ev[4]);
    t.kernel_launches = 4;
    t.h2d_bytes = h2d;
    t.d2h_bytes = (uint64_t) n * sizeof(DevRec);
    int worst = UNC_OK;
    for (uint32_t i = 0; i < n; i++) if (out[i].status != 0) worst = UNC_E_OVERFLOW;
    if (worst) return fail(worst, "a read overflowed its seed-cluster workspace (see unc_paf_rec.status)");
    return UNC_OK;
}

static int run_batch(unc_pool *P, const unc_read_desc *reads, uint32_t n, const void *samples, bool on_device,
                     unc_paf_rec *out) {
    if (!out) return fail(UNC_E_ARG, "null argument");
    int rc = batch_enqueue(P, reads, n, samples, on_device);
    if (rc) return rc;
    return batch_finish(P, out);
}

int unc_map_batch(unc_pool *P, const unc_read_desc *reads, uint32_t n, const void *samples, unc_paf_rec *out) {
    return run_batch(P, reads, n, samples, false, out);
}

int unc_map_batch_submit(unc_pool *P, const unc_read_desc *reads, uint32_t n, const void *samples, int samples_on_device) {
    return batch_enqueue(P, reads, n, samples, samples_on_device != 0);
}

int unc_map_batch_wait(unc_pool *P, unc_paf_rec *out) {
    return batch_finish(P, out);
}

int unc_pool_record(unc_pool *P, int slot) {
    if (!P || slot < 0 || slot > 1) return fail(UNC_E_ARG, "bad argument");
    CUDA_TRY(cudaSetDevice(P->idx->device));
    if (!P->ev_user[slot]) CUDA_TRY(cudaEventCreate(&P->ev_user[slot]));
    CUDA_TRY(cudaEventRecord(P->ev_user[slot], P->stream));
    return UNC_OK;
}

int unc_pool_elapsed(unc_pool *from, int from_slot, unc_pool *to, int to_slot, float *ms) {
    if (!from || !to || !ms || from_slot < 0 || from_slot > 1 || to_slot < 0 || to_slot > 1 || !from->ev_user[from_slot] ||
        !to->ev_user[to_slot])
        return fail(UNC_E_ARG, "bad argument or event never recorded");
    CUDA_TRY(cudaSetDevice(to->idx->device));
    CUDA_TRY(cudaEventSynchronize(from->ev_user[from_slot]));
    CUDA_TRY(cudaEventSynchronize(to->ev_user[to_slot]));
    CUDA_TRY(cudaEventElapsedTime(ms, from->ev_user[from_slot], to->ev_user[to_slot]));
    return UNC_OK;
}

int unc_map_batch_device(unc_pool *P, const unc_read_desc *reads, uint32_t n, const void *d_samples, unc_paf_rec *out) {
    return run_batch(P, reads, n, d_samples, true, out);
}

int unc_pool_set_tie_order(unc_pool *P, int mode) {
    if (!P || (mode != 0 && mode != 1)) return fail(UNC_E_ARG, "bad argument");
    if (P->pending_n) return fail(UNC_E_ARG, "the pool holds a submitted batch");
    if (mode == 1) {
        CUDA_TRY(cudaSetDevice(P->idx->device));
        CUDA_TRY(raise_dyn_smem(k2_map_exact, P->smem));
        // CTAs are independent (each pulls reads from the queue into its own slot), so a lower residency than k2_map's
        // only means that the last CTAs of the grid start late and find the queue empty
    }
    P->tie_order = mode;
    return UNC_OK;
}

int unc_map_batch_ordered(unc_pool *P, const unc_read_desc *reads, uint32_t n, const void *samples, int samples_on_device,
                          uint32_t carry[32], unc_paf_rec *out, uint32_t *n_remapped, uint32_t *n_rounds) {
    if (!P || !reads || !samples || !carry || !out) return fail(UNC_E_ARG, "null argument");
    if (n == 0 || n > P->max_reads) return fail(UNC_E_ARG, "n_reads outside 1..max_reads");
    bool first = true;
    unc_timing sum;
    memset(&sum, 0, sizeof(sum));
    std::vector<unc_read_desc> sub;
    auto map_subset = [&](const uint32_t *ids, uint32_t m, const uint32_t *fi, uint32_t *fo, unc_paf_rec *recs, uint32_t *cand) -> int {
        sub.resize(m);
        for (uint32_t j = 0; j < m; j++) sub[j] = reads[ids[j]];
        // after round 0 the samples are on the device (the pool's staging buffer, or where the caller put them)
        const void *src = first ? samples : (samples_on_device ? samples : (const void *) P->d_samples);
        P->want_cand = cand != nullptr;
        int rc = batch_enqueue(P, sub.data(), m, src, first ? samples_on_device != 0 : true, fi);
        P->want_cand = false;
        first = false;
        if (rc) return rc;
        rc = batch_finish(P, recs);
        if (rc != UNC_OK && rc != UNC_E_OVERFLOW) return rc;
        CUDA_TRY(cudaMemcpy(fo, P->d_flags_out, (size_t) m * 128, cudaMemcpyDeviceToHost));
        if (cand) CUDA_TRY(cudaMemcpy(cand, P->d_cand, (size_t) m * 128, cudaMemcpyDeviceToHost));
        const unc_timing &t = P->last;
        sum.h2d_ms += t.h2d_ms; sum.k1_ms += t.k1_ms; sum.k1_events_ms += t.k1_events_ms; sum.k2_ms += t.k2_ms;
        sum.d2h_ms += t.d2h_ms; sum.total_ms += t.total_ms; sum.kernel_launches += t.kernel_launches + (cand ? 1u : 0u);
        sum.h2d_bytes += t.h2d_bytes; sum.d2h_bytes += t.d2h_bytes + (uint64_t) m * (cand ? 256 : 128);
        return rc;
    };
    int rc = unc_ordered_map(n, P->prm.max_paths, carry, out, n_remapped, n_rounds, map_subset);
    P->last = sum;
    if (rc == UNC_E_OVERFLOW) return fail(rc, "a read overflowed its seed-cluster workspace (see unc_paf_rec.status)");
    return rc;
}

int unc_events_batch(unc_pool *P, const unc_read_desc *reads, uint32_t n, const void *samples, uint32_t stride,
                     float *events, float *normed, uint32_t *n_events, float *mean_event_len) {
    if (!P || !reads || !samples) return fail(UNC_E_ARG, "null argument");
    if (P->pending_n) return fail(UNC_E_ARG, "the pool holds a submitted batch (its staging buffers are in use): call unc_map_batch_wait first");
    CUDA_TRY(cudaSetDevice(P->idx->device));
    uint64_t span = 0;
    uint32_t mx = 0;
    int rc = stage_reads(P, reads, n, &span, &mx, true);
    if (rc) return rc;
    if (stride < mx) return fail(UNC_E_ARG, "stride smaller than the longest read");
    cudaStream_t s = P->stream;
    CUDA_TRY(cudaEventRecord(P->ev[0], s));
    CUDA_TRY(cudaMemcpyAsync(P->d_samples, samples, span, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(P->d_reads, P->h_reads, (size_t) n * sizeof(DevReadDesc), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaEventRecord(P->ev[1], s));
    CUDA_TRY(cudaMemsetAsync(P->d_queue, 0, 32, s));
    DevBatch B = make_batch(P, P->d_samples, (span + 15) & ~(uint64_t) 15, n, true);
    launch_k1(P, B, n, s);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(P->ev[2], s));
    CUDA_TRY(cudaStreamSynchronize(s));
    std::vector<uint32_t> ne(n);
    CUDA_TRY(cudaMemcpy(ne.data(), P->d_n_events, (size_t) n * 4, cudaMemcpyDeviceToHost));
    if (n_events) memcpy(n_events, ne.data(), (size_t) n * 4);
    if (mean_event_len) CUDA_TRY(cudaMemcpy(mean_event_len, P->d_mel, (size_t) n * 4, cudaMemcpyDeviceToHost));
    if (events)
        CUDA_TRY(cudaMemcpy2D(events, (size_t) stride * 4, P->d_events, (size_t) P->ev_stride * 4, (size_t) mx * 4, n,
                              cudaMemcpyDeviceToHost));
    if (normed)
        CUDA_TRY(cudaMemcpy2D(normed, (size_t) stride * 4, P->d_normed, (size_t) P->ev_stride * 4, (size_t) mx * 4, n,
                              cudaMemcpyDeviceToHost));
    unc_timing &t = P->last;
    memset(&t, 0, sizeof(t));
    cudaEventElapsedTime(&t.h2d_ms, P->ev[0], P->ev[1]);
    cudaEventElapsedTime(&t.k1_ms, P->ev[1], P->ev[2]);
    cudaEventElapsedTime(&t.k1_events_ms, P->ev[1], P->ev[5]);
    t.total_ms = t.h2d_ms + t.k1_ms;
    t.kernel_launches = 3;
    t.h2d_bytes = span + (uint64_t) n * sizeof(DevReadDesc);
    return UNC_OK;
}

int unc_match_probs(const unc_index *x, float event, float out[1024]) {
    if (!x || !out) return fail(UNC_E_ARG, "null argument");
    CUDA_TRY(cudaSetDevice(x->device));
    float *d = nullptr;
    CUDA_TRY(cudaMalloc(&d, 1024 * 4));
    k_match_probs<<<4, 256>>>(x->ix, event, d);
    cudaError_t e = cudaMemcpy(out, d, 1024 * 4, cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) return fail(UNC_E_CUDA, cudaGetErrorString(e));
    return UNC_OK;
}

int unc_fm_neighbors(const unc_index *x, uint32_t n, const uint64_t *start, const uint64_t *end, const uint8_t *base,
                     uint64_t *ostart, uint64_t *oend) {
    if (!x || !n) return fail(UNC_E_ARG, "null argument");
    CUDA_TRY(cudaSetDevice(x->device));
    u64 *ds, *de, *dos, *doe;
    u8 *db;
    CUDA_TRY(cudaMalloc(&ds, n * 8)); CUDA_TRY(cudaMalloc(&de, n * 8)); CUDA_TRY(cudaMalloc(&dos, n * 8));
    CUDA_TRY(cudaMalloc(&doe, n * 8)); CUDA_TRY(cudaMalloc(&db, n));
    cudaMemcpy(ds, start, n * 8, cudaMemcpyHostToDevice);
    cudaMemcpy(de, end, n * 8, cudaMemcpyHostToDevice);
    cudaMemcpy(db, base, n, cudaMemcpyHostToDevice);
    k_fm_neighbors<<<(n + 127) / 128, 128>>>(x->ix, n, ds, de, db, dos, doe);
    cudaMemcpy(ostart, dos, n * 8, cudaMemcpyDeviceToHost);
    cudaError_t e = cudaMemcpy(oend, doe, n * 8, cudaMemcpyDeviceToHost);
    cudaFree(ds); cudaFree(de); cudaFree(dos); cudaFree(doe); cudaFree(db);
    if (e != cudaSuccess) return fail(UNC_E_CUDA, cudaGetErrorString(e));
    return UNC_OK;
}

int unc_fm_sa(const unc_index *x, uint32_t n, const uint64_t *rows, uint64_t *out) {
    if (!x || !n) return fail(UNC_E_ARG, "null argument");
    CUDA_TRY(cudaSetDevice(x->device));
    u64 *dr, *dout;
    CUDA_TRY(cudaMalloc(&dr, n * 8)); CUDA_TRY(cudaMalloc(&dout, n * 8));
    cudaMemcpy(dr, rows, n * 8, cudaMemcpyHostToDevice);
    k_fm_sa<<<(n + 127) / 128, 128>>>(x->ix, n, dr, dout);
    cudaError_t e = cudaMemcpy(out, dout, n * 8, cudaMemcpyDeviceToHost);
    cudaFree(dr); cudaFree(dout);
    if (e != cudaSuccess) return fail(UNC_E_CUDA, cudaGetErrorString(e));
    return UNC_OK;
}

// debug builds (-DUNC_PHASE_TIMING): per-read cycle counters of the mapper's phases
int unc_pool_debug_phases(const unc_pool *P, uint32_t n, unsigned long long *out) {
    if (!P || !out || !P->d_dbg) return fail(UNC_E_ARG, "phase timing not compiled in");
    CUDA_TRY(cudaMemcpy(out, P->d_dbg, (size_t) n * 512, cudaMemcpyDeviceToHost));
    return UNC_OK;
}
// ... and the timeline of read UNC_PT_TRACE_READ of a batch of n reads: [event][warp][mark] clock values (UNC_PT_TRACE_BYTES)
int unc_pool_debug_trace(const unc_pool *P, uint32_t n, unsigned long long *out) {
    if (!P || !out || !P->d_dbg) return fail(UNC_E_ARG, "phase timing not compiled in");
#ifdef UNC_PHASE_TIMING
    CUDA_TRY(cudaMemcpy(out, P->d_dbg + (size_t) n * 64, UNC_PT_TRACE_BYTES, cudaMemcpyDeviceToHost));
#endif
    return UNC_OK;
}

int unc_pool_k1_stats(const unc_pool *P, uint32_t out[4]) {
    if (!P || !out) return fail(UNC_E_ARG, "null argument");
    if (P->pending_n) return fail(UNC_E_ARG, "the pool holds a submitted batch: call unc_map_batch_wait first");
    CUDA_TRY(cudaMemcpy(out, P->d_queue + 2, 16, cudaMemcpyDeviceToHost));
    return UNC_OK;
}

int unc_pool_last_timing(const unc_pool *P, unc_timing *t) {
    if (!P || !t) return fail(UNC_E_ARG, "null argument");
    *t = P->last;
    return UNC_OK;
}

}  // extern "C"

#include "unc_stream_host.inl"
#include "unc_selfalign_host.inl"
#include "unc_dtw_host.inl"
