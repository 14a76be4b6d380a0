// msda_cabi.cu -- the C ABI declared in include/msda_b200.h: argument checks, kernel routing, launches.
// Replaces the reference host wrappers ms_deform_attn_cuda_forward/backward (ops/src/cuda/ms_deform_attn_cuda.cu)
// and launchers ms_deformable_im2col_cuda / ms_deformable_col2im_cuda (ms_deform_im2col_cuda.cuh:923-954,956-1327).
#include <atomic>
#include <cstdio>
#include <cstdlib>

#include "../../include/msda_b200.h"
#include "msda_condinst.cuh"
#include "msda_generic.cuh"
#include "msda_module.cuh"
#include "msda_slab.cuh"
#include "msda_tmem.cuh"
#include "msda_tiled.cuh"

namespace {

std::atomic<uint64_t> g_launches{0};

struct Dims { int N, S, M, D, L, Lq, P; };

inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int check_dims(const Dims &d) {
    if (d.N <= 0 || d.S <= 0 || d.M <= 0 || d.D <= 0 || d.L <= 0 || d.Lq <= 0 || d.P <= 0) return MSDA_E_BADARG;
    // rows are indexed with int32 inside a batch element; tap counts with int64 everywhere.
    if ((long long)d.S >= (1ll << 30)) return MSDA_E_TOOLARGE;
    if ((long long)d.N * d.Lq * d.M >= (1ll << 40)) return MSDA_E_TOOLARGE;
    return 0;
}

// Per-device caches (a process may drive several GPUs: SM counts, occupancy and function attributes are per device).
constexpr int kMaxDevices = 64;

int current_device() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) dev = 0;
    return dev;
}

int num_sms() {
    static std::atomic<int> sms[kMaxDevices];
    const int dev = current_device();
    int v = sms[dev].load(std::memory_order_relaxed);
    if (v == 0) {
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
        sms[dev].store(v, std::memory_order_relaxed);
    }
    return v;
}

int env_int(const char *name, int dflt) {
    const char *e = getenv(name);
    return (e && e[0]) ? atoi(e) : dflt;
}

// Kernel-selection knobs (msda_set_knob): environment defaults, overridable at run time.  g_knob_epoch invalidates the
// per-device launch configurations derived from them.
struct Knobs {
    std::atomic<int> v[MSDA_KNOB_COUNT];
    std::atomic<int> epoch{1};
    Knobs() {
        v[MSDA_KNOB_SLAB].store(env_int("MSDA_SLAB", -1));
        v[MSDA_KNOB_BWD_WIN_ROWS].store(env_int("MSDA_BWD_WIN_ROWS", -1));
        v[MSDA_KNOB_BWD_LIST_CAP].store(env_int("MSDA_BWD_LIST_CAP", 48));
        v[MSDA_KNOB_FWD_SLAB_CTAS].store(env_int("MSDA_FWD_SLAB_CTAS", 2));
        v[MSDA_KNOB_F32_VEC8_FWD].store(env_int("MSDA_F32_VEC8_FWD", 0));
        v[MSDA_KNOB_F32_VEC8_BWD].store(env_int("MSDA_F32_VEC8_BWD", 0));
        v[MSDA_KNOB_BF16_FINE_ROWS].store(env_int("MSDA_BF16_FINE_ROWS", 0));
        v[MSDA_KNOB_BF16_PACKED_FWD].store(env_int("MSDA_BF16_PACKED_FWD", 0));
        v[MSDA_KNOB_ZERO_FILL].store(env_int("MSDA_ZERO_FILL", 2));   // measured: profiles/r02zy_zero_fill_ab.txt
    }
};
Knobs &knobs() { static Knobs k; return k; }
int knob(int i) { return knobs().v[i].load(std::memory_order_relaxed); }

// Set by msda_backward_* when the zero-fill just issued on the stream may be the PDL primary of the next launch; consumed
// (and cleared) by launch_bwd, cleared by msda_backward_* on every other route.
thread_local bool t_pdl_next = false;

// Zero-fill of grad_value before the backward kernels (MSDA_KNOB_ZERO_FILL).  *pdl is set when the fill went out as a
// kernel that the NEXT launch on `st` may take as its programmatic-dependent-launch primary.  The fill kernel stands in
// for a memset and is not counted by msda_launch_count().
cudaError_t zero_fill(void *p, size_t bytes, cudaStream_t st, bool *pdl = nullptr) {
    if (pdl) *pdl = false;
    const int mode = knob(MSDA_KNOB_ZERO_FILL);
    if (mode <= 0 || bytes < (1u << 16) || !aligned16(p) || (bytes & 15u)) return cudaMemsetAsync(p, 0, bytes, st);
    const unsigned long long n16 = bytes >> 4;
    unsigned long long blocks = (n16 + 255) / 256;
    const unsigned long long wave = (unsigned long long)num_sms() * 8;       // 8 x 256 threads = every thread slot of an SM
    if (blocks > wave) blocks = wave;
    msda::msda_zero_fill<<<(unsigned)blocks, 256, 0, st>>>(static_cast<uint4 *>(p), n16);
    const cudaError_t err = cudaGetLastError();
    if (pdl && mode >= 2 && err == cudaSuccess) {
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        *pdl = cudaStreamIsCapturing(st, &cap) == cudaSuccess && cap == cudaStreamCaptureStatusNone;
    }
    return err;
}

// ---- routing ------------------------------------------------------------------------------------------------
// Fast path: D in {16,32,64} (fp32) / {32,64} (bf16), L <= kMaxLevels, L*P <= 32.  LP_MAX is the compile-time tap
// capacity (taps beyond L*P are dead: zero weight, row 0).
bool fast_ok(int dtype_bytes, int D, int L, int P) {
    if (L > msda::kMaxLevels || L * P > 32) return false;
    if (dtype_bytes == 4) return D == 16 || D == 32 || D == 64;
    if (dtype_bytes == 2) return D == 32 || D == 64;
    return false;
}

bool use_fast(int dtype_bytes, const Dims &d) {      // the tiled kernels index (b,q,m) pairs with 31 bits
    return fast_ok(dtype_bytes, d.D, d.L, d.P) && (long long)d.N * d.Lq * d.M < (1ll << 31);
}

// Persistent launch: one CTA per resident slot (SM count x occupancy); tiles are walked with a grid stride inside the
// kernel, which derives the tile map from the device-resident level table (no host read of spatial_shapes).
template <typename K>
int resident_ctas(K kernel) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, msda::kTiledThreads, 0) != cudaSuccess || per_sm < 1)
        per_sm = 1;
    return per_sm * num_sms();
}

// resident_ctas() cached per (kernel instantiation, device)
template <typename K>
int resident_ctas_cached(K kernel, std::atomic<int> (&cache)[kMaxDevices]) {
    const int dev = current_device();
    int v = cache[dev].load(std::memory_order_relaxed);
    if (v == 0) { v = resident_ctas(kernel); cache[dev].store(v, std::memory_order_relaxed); }
    return v;
}

// Slot order.  Measured on B200 (profiles/r01c_*_ncu.md, gpurun_out r01d sweep): the 8x8-pixel patch order lifts the
// forward L1 sector hit rate from 39% to 75% and cuts L2 traffic 2.4x, but the kernels are bound by the LSU's
// global-load issue rate (~7.5 cycles per 512-byte LDG.128 per SM), not by L1 misses, so run time does not move while
// partially filled border patches cost 7-15% idle slots.  Linear order is therefore the default; MSDA_PATCHES=1
// re-enables the patch order for experiments.
int allow_patches() {
    static int v = -1;
    if (v < 0) { const char *e = getenv("MSDA_PATCHES"); v = (e && e[0] == '1') ? 1 : 0; }
    return v;
}

// TMA staging of (x, y, a): linear slot order only, and every pair's tap run must start 16-byte aligned (L*P % 4 == 0).
// MSDA_NO_TMA=1 switches it off (A/B measurements).
bool use_tma_staging(const Dims &d) {
    static int off = -1;
    if (off < 0) { const char *e = getenv("MSDA_NO_TMA"); off = (e && e[0] == '1') ? 1 : 0; }
    return !off && !allow_patches() && ((d.L * d.P) % 4 == 0);
}

// Small launches (decoder-style calls: a few thousand pairs) cannot hide the row-load latency with other warps; there the
// taps of each pair are split over the groups of a warp (template SPLIT).  MSDA_SPLIT=0/1 forces the choice (A/B).
bool use_split(unsigned npairs) {
    static int force = -2;
    if (force == -2) { const char *e = getenv("MSDA_SPLIT"); force = (e && (e[0] == '0' || e[0] == '1')) ? e[0] - '0' : -1; }
    if (force >= 0) return force == 1;
    // measured (gpurun r01p): 4 800 pairs (cfg2 decoder call) fwd 18.4 -> 14.4 us, bwd 29.7 -> 27.6 us; neutral-to-worse
    // from 14 400 pairs up, so only launches with fewer than ~56 pairs per SM are split
    return npairs <= (unsigned)num_sms() * 56u;
}

constexpr int kFwdMinCtas = 4, kBwdMinCtas = 2;     // r01d sweep: fwd flat for 3..5, bwd best at 2 (128 regs, no spills)


template <typename T> struct FwdVec { static constexpr int v = 16 / sizeof(T); };      // 16-byte row slices
template <typename T> struct BwdVec { static constexpr int v = 4; };                  // 4 channels per lane (see RowVec)

template <typename T, int D, int LP_MAX, int VEC = FwdVec<T>::v>
cudaError_t launch_fwd(const T *value, const int64_t *shapes, const int64_t *lsi, const float *loc, const float *attn,
                       const Dims &d, T *out, cudaStream_t st) {
    constexpr int GPW = 32 / (D / VEC);
    constexpr bool kCanStage = (LP_MAX <= 16);          // per-warp double buffer must fit static shared memory
    constexpr bool kCanSplit = (LP_MAX % GPW == 0) && (LP_MAX / GPW <= D / VEC);
    const unsigned npairs = (unsigned)((long long)d.N * d.Lq * d.M);
    const bool split = kCanSplit && use_split(npairs);
    const bool tma = !split && kCanStage && use_tma_staging(d);
    if constexpr (sizeof(T) == 2 && VEC == 8) {      // bf16: packed-bf16 corner blend for the large (non-split) launches
        if (!split && knob(MSDA_KNOB_BF16_PACKED_FWD) == 1) {
            static std::atomic<int> c_ptma[kMaxDevices], c_pldg[kMaxDevices];
            auto k_tma = msda::msda_fwd_tiled<T, VEC, D, LP_MAX, kFwdMinCtas, kCanStage, false, true>;
            auto k_ldg = msda::msda_fwd_tiled<T, VEC, D, LP_MAX, kFwdMinCtas, false, false, true>;
            const int pslots = tma ? resident_ctas_cached(k_tma, c_ptma) : resident_ctas_cached(k_ldg, c_pldg);
            const unsigned ip = msda::kTiledWarps * GPW;
            const unsigned tub = (npairs + ip - 1) / ip;
            const int pgrid = (int)(tub < (unsigned)pslots ? tub : (unsigned)pslots);
            (tma ? k_tma : k_ldg)<<<pgrid, msda::kTiledThreads, 0, st>>>(value, shapes, lsi, loc, attn, d.N, d.S, d.M, d.L, d.Lq, d.P,
                                                                          npairs, allow_patches(), out);
            g_launches.fetch_add(1, std::memory_order_relaxed);
            return cudaGetLastError();
        }
    }
    auto kern = split ? msda::msda_fwd_tiled<T, VEC, D, LP_MAX, kFwdMinCtas, false, kCanSplit>
                : tma ? msda::msda_fwd_tiled<T, VEC, D, LP_MAX, kFwdMinCtas, kCanStage, false>
                      : msda::msda_fwd_tiled<T, VEC, D, LP_MAX, kFwdMinCtas, false, false>;
    static std::atomic<int> c_split[kMaxDevices], c_tma[kMaxDevices], c_ldg[kMaxDevices];
    const int slots = split ? resident_ctas_cached(msda::msda_fwd_tiled<T, VEC, D, LP_MAX, kFwdMinCtas, false, kCanSplit>, c_split)
                      : tma ? resident_ctas_cached(msda::msda_fwd_tiled<T, VEC, D, LP_MAX, kFwdMinCtas, kCanStage, false>, c_tma)
                            : resident_ctas_cached(msda::msda_fwd_tiled<T, VEC, D, LP_MAX, kFwdMinCtas, false, false>, c_ldg);
    const unsigned iter_pairs = msda::kTiledWarps * (split ? 1 : GPW);
    const unsigned tiles_ub = (npairs + iter_pairs - 1) / iter_pairs;        // linear order (patch order has fewer, larger tiles)
    const int grid = (int)(tiles_ub < (unsigned)slots ? tiles_ub : (unsigned)slots);
    kern<<<grid, msda::kTiledThreads, 0, st>>>(value, shapes, lsi, loc, attn, d.N, d.S, d.M, d.L, d.Lq, d.P, npairs,
                                               allow_patches(), out);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}

template <typename T, int D, int LP_MAX, int VEC = BwdVec<T>::v, bool DET = false>
cudaError_t launch_bwd(const T *grad_out, const T *value, const int64_t *shapes, const int64_t *lsi, const float *loc,
                       const float *attn, const Dims &d, float *gv, float *gl, float *ga, cudaStream_t st,
                       unsigned long long *det_acc, int det_clog2) {
    constexpr int GPW = 32 / (D / VEC);
    constexpr bool kCanStage = (LP_MAX <= 16);
    constexpr bool kCanSplit = (LP_MAX % GPW == 0) && (LP_MAX / GPW <= D / VEC);
    const unsigned npairs = (unsigned)((long long)d.N * d.Lq * d.M);
    const bool split = kCanSplit && use_split(npairs);
    const bool tma = !split && kCanStage && use_tma_staging(d);
    auto kern = split ? msda::msda_bwd_tiled<T, VEC, D, LP_MAX, kBwdMinCtas, false, kCanSplit, false, DET>
                : tma ? msda::msda_bwd_tiled<T, VEC, D, LP_MAX, kBwdMinCtas, kCanStage, false, false, DET>
                      : msda::msda_bwd_tiled<T, VEC, D, LP_MAX, kBwdMinCtas, false, false, false, DET>;
    static std::atomic<int> c_split[kMaxDevices], c_tma[kMaxDevices], c_ldg[kMaxDevices];
    const int slots = split ? resident_ctas_cached(msda::msda_bwd_tiled<T, VEC, D, LP_MAX, kBwdMinCtas, false, kCanSplit, false, DET>, c_split)
                      : tma ? resident_ctas_cached(msda::msda_bwd_tiled<T, VEC, D, LP_MAX, kBwdMinCtas, kCanStage, false, false, DET>, c_tma)
                            : resident_ctas_cached(msda::msda_bwd_tiled<T, VEC, D, LP_MAX, kBwdMinCtas, false, false, false, DET>, c_ldg);
    const unsigned iter_pairs = msda::kTiledWarps * (split ? 1 : GPW);
    const unsigned tiles_ub = (npairs + iter_pairs - 1) / iter_pairs;
    const int grid = (int)(tiles_ub < (unsigned)slots ? tiles_ub : (unsigned)slots);
    const bool pdl = t_pdl_next;
    t_pdl_next = false;
    if (pdl) {       // the preceding launch on `st` is msda_zero_fill(grad_value): let this kernel's prologue overlap it
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)grid);
        cfg.blockDim = dim3(msda::kTiledThreads);
        cfg.dynamicSmemBytes = 0;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, grad_out, value, shapes, lsi, loc, attn, d.N, d.S, d.M, d.L, d.Lq,
                                                 d.P, npairs, allow_patches(), gv, gl, ga, (__nv_bfloat16 *)nullptr, 0,
                                                 det_acc, det_clog2);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        return e != cudaSuccess ? e : cudaGetLastError();
    }
    kern<<<grid, msda::kTiledThreads, 0, st>>>(grad_out, value, shapes, lsi, loc, attn, d.N, d.S, d.M, d.L, d.Lq, d.P,
                                               npairs, allow_patches(), gv, gl, ga, nullptr, 0, det_acc, det_clog2);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}

// ---- slab-ordered kernels (msda_slab.cuh): D = 32 and L*P <= 16 (every UNINEXT call) ------------------------------
// OPT-IN (MSDA_KNOB_SLAB = 1).  Measured at cfg2 (gpurun r02c, profiles/r02c_slab_kernels_ncu.md): forward 0.186 ms against
// 0.175 ms tiled although L2 sectors halve and the L1 hit rate doubles; backward 0.654 ms against 0.480 ms although red
// sectors drop 43 % -- the shared-memory traffic of the window (4 wavefronts per privatised row-add) lands on the same
// LSU data pipe that the gathers already keep > 50 % busy.  MSDA_KNOB_SLAB = -1 (auto) therefore selects the tiled kernels.

bool use_slab(const Dims &d, unsigned npairs, const void *value, const void *out) {
    if (d.D != 32 || d.L * d.P > 16 || d.L > msda::kMaxLevels) return false;
    if ((reinterpret_cast<uintptr_t>(value) & 31u) || (reinterpret_cast<uintptr_t>(out) & 15u)) return false;   // LDG.256 rows
    (void)npairs;
    return knob(MSDA_KNOB_SLAB) == 1;
}

template <typename T>
cudaError_t launch_fwd_slab(const T *value, const int64_t *shapes, const int64_t *lsi, const float *loc, const float *attn,
                            const Dims &d, T *out, cudaStream_t st) {
    const int ctas_per_sm = knob(MSDA_KNOB_FWD_SLAB_CTAS) == 1 ? 1 : 2;
    const int sms = num_sms();
    if (ctas_per_sm == 2)
        msda::msda_fwd_slab<T, 16, 2><<<sms * 2, msda::kSlabThreads, 0, st>>>(value, shapes, lsi, loc, attn, d.N, d.S, d.M, d.L,
                                                                              d.Lq, d.P, sms, out);
    else
        msda::msda_fwd_slab<T, 16, 1><<<sms, msda::kSlabThreads, 0, st>>>(value, shapes, lsi, loc, attn, d.N, d.S, d.M, d.L,
                                                                          d.Lq, d.P, sms, out);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_bwd_slab(const T *grad_out, const T *value, const int64_t *shapes, const int64_t *lsi, const float *loc,
                            const float *attn, const Dims &d, float *gv, float *gl, float *ga, cudaStream_t st) {
    // shared-memory budget: the opt-in maximum of the device minus the kernel's static part; the window gets what the
    // lists / g stash / tap slabs leave.  MSDA_BWD_WIN_ROWS / MSDA_BWD_LIST_CAP override (sweeps).
    static std::atomic<int> win_rows[kMaxDevices], cap_c[kMaxDevices], epoch_c[kMaxDevices];
    const int dev = current_device();
    const int epoch = knobs().epoch.load(std::memory_order_acquire);
    int rows = win_rows[dev].load(std::memory_order_relaxed), cap = cap_c[dev].load(std::memory_order_relaxed);
    auto kern = msda::msda_bwd_slab<T, 16>;
    if (rows == 0 || epoch_c[dev].load(std::memory_order_relaxed) != epoch) {
        int max_optin = 0;
        cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        cudaFuncAttributes fa{};
        cudaFuncGetAttributes(&fa, kern);
        cap = knob(MSDA_KNOB_BWD_LIST_CAP) & ~1;
        if (cap < 8) cap = 8;
        const long long fixed = (long long)msda::bwd_slab_smem_bytes(0, cap) + (long long)fa.sharedSizeBytes + 64;
        rows = (int)((max_optin - fixed) / 128);
        const int want = knob(MSDA_KNOB_BWD_WIN_ROWS);
        if (want >= 0 && want < rows) rows = want;
        if (rows < 0) rows = 0;
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)msda::bwd_slab_smem_bytes(rows, cap));
        if (e != cudaSuccess) return e;
        cap_c[dev].store(cap, std::memory_order_relaxed);
        win_rows[dev].store(rows == 0 ? -1 : rows, std::memory_order_relaxed);
        epoch_c[dev].store(epoch, std::memory_order_relaxed);
    }
    if (rows < 0) rows = 0;
    const int sms = num_sms();
    kern<<<sms, msda::kSlabThreads, msda::bwd_slab_smem_bytes(rows, cap), st>>>(grad_out, value, shapes, lsi, loc, attn, d.N,
                                                                               d.S, d.M, d.L, d.Lq, d.P, sms, rows, cap, gv,
                                                                               gl, ga);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}

// bf16 backward with the fine levels accumulated in the bf16 result (msda_bwd_tiled MIXED): D = 32, L*P <= 16, large launches.
cudaError_t launch_bwd_mixed(const __nv_bfloat16 *go, const __nv_bfloat16 *value, const int64_t *shapes, const int64_t *lsi,
                             const float *loc, const float *attn, const Dims &d, float *scratch, __nv_bfloat16 *gv16,
                             float *gl, float *ga, int fine_min_rows, cudaStream_t st) {
    using T = __nv_bfloat16;
    constexpr int VEC = 4, DD = 32, LP_MAX = 16;
    constexpr int GPW = 32 / (DD / VEC);
    const unsigned npairs = (unsigned)((long long)d.N * d.Lq * d.M);
    const bool tma = use_tma_staging(d);
    static std::atomic<int> c_tma[kMaxDevices], c_ldg[kMaxDevices];
    auto k_tma = msda::msda_bwd_tiled<T, VEC, DD, LP_MAX, kBwdMinCtas, true, false, true>;
    auto k_ldg = msda::msda_bwd_tiled<T, VEC, DD, LP_MAX, kBwdMinCtas, false, false, true>;
    const int slots = tma ? resident_ctas_cached(k_tma, c_tma) : resident_ctas_cached(k_ldg, c_ldg);
    const unsigned iter_pairs = msda::kTiledWarps * GPW;
    const unsigned tiles_ub = (npairs + iter_pairs - 1) / iter_pairs;
    const int grid = (int)(tiles_ub < (unsigned)slots ? tiles_ub : (unsigned)slots);
    (tma ? k_tma : k_ldg)<<<grid, msda::kTiledThreads, 0, st>>>(go, value, shapes, lsi, loc, attn, d.N, d.S, d.M, d.L, d.Lq,
                                                                 d.P, npairs, allow_patches(), scratch, gl, ga, gv16,
                                                                 fine_min_rows, nullptr, 0);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}

// Backward with tensor-memory accumulators for the coarse levels (msda_tmem.cuh): MSDA_KNOB_SLAB = 2.
template <typename T>
cudaError_t launch_bwd_tmem(const T *grad_out, const T *value, const int64_t *shapes, const int64_t *lsi, const float *loc,
                            const float *attn, const Dims &d, float *gv, float *gl, float *ga, cudaStream_t st) {
    static std::atomic<int> ready[kMaxDevices], cap_c[kMaxDevices], epoch_c[kMaxDevices];
    const int dev = current_device();
    const int epoch = knobs().epoch.load(std::memory_order_acquire);
    auto kern = msda::msda_bwd_tmem<T, 16>;
    int cap = cap_c[dev].load(std::memory_order_relaxed);
    if (!ready[dev].load(std::memory_order_relaxed) || epoch_c[dev].load(std::memory_order_relaxed) != epoch) {
        cap = knob(MSDA_KNOB_BWD_LIST_CAP) & ~1;
        if (cap < 8) cap = 8;
        if (cap > 128) cap = 128;
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msda::bwd_tmem_smem_bytes(cap));
        if (e != cudaSuccess) return e;
        cap_c[dev].store(cap, std::memory_order_relaxed);
        epoch_c[dev].store(epoch, std::memory_order_relaxed);
        ready[dev].store(1, std::memory_order_relaxed);
    }
    const int sms = num_sms();
    kern<<<sms, msda::kTmThreads, msda::bwd_tmem_smem_bytes(cap), st>>>(grad_out, value, shapes, lsi, loc, attn, d.N, d.S, d.M, d.L,
                                                                        d.Lq, d.P, sms, cap, gv, gl, ga);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}

#define MSDA_ROUTE_LP(T, DD, CALL)                                   \
    (LP <= 16 ? CALL<T, DD, 16> : CALL<T, DD, 32>)

template <typename T>
cudaError_t fwd_fast(const T *value, const int64_t *shapes, const int64_t *lsi, const float *loc, const float *attn,
                     const Dims &d, T *out, cudaStream_t st) {
    const int LP = d.L * d.P;
    if (use_slab(d, (unsigned)((long long)d.N * d.Lq * d.M), value, out))
        return launch_fwd_slab<T>(value, shapes, lsi, loc, attn, d, out, st);
    if constexpr (sizeof(T) == 4) {           // fp32, 32-byte lanes (LDG.256): needs 32-byte aligned rows
        if (knob(MSDA_KNOB_F32_VEC8_FWD) == 1 && LP <= 16 && (d.D == 32 || d.D == 64) &&
            !(reinterpret_cast<uintptr_t>(value) & 31u))
            return d.D == 32 ? launch_fwd<T, 32, 16, 8>(value, shapes, lsi, loc, attn, d, out, st)
                             : launch_fwd<T, 64, 16, 8>(value, shapes, lsi, loc, attn, d, out, st);
    }
    switch (d.D) {
        case 16: if constexpr (sizeof(T) == 4) return MSDA_ROUTE_LP(T, 16, launch_fwd)(value, shapes, lsi, loc, attn, d, out, st); break;
        case 32: return MSDA_ROUTE_LP(T, 32, launch_fwd)(value, shapes, lsi, loc, attn, d, out, st);
        case 64: return MSDA_ROUTE_LP(T, 64, launch_fwd)(value, shapes, lsi, loc, attn, d, out, st);
    }
    return cudaErrorInvalidValue;
}

template <typename T>
cudaError_t bwd_fast(const T *go, const T *value, const int64_t *shapes, const int64_t *lsi, const float *loc,
                     const float *attn, const Dims &d, float *gv, float *gl, float *ga, cudaStream_t st) {
    const int LP = d.L * d.P;
    if (knob(MSDA_KNOB_SLAB) == 2 && d.D == 32 && LP <= 16 && d.L <= msda::kMaxLevels)
        return launch_bwd_tmem<T>(go, value, shapes, lsi, loc, attn, d, gv, gl, ga, st);
    if (use_slab(d, (unsigned)((long long)d.N * d.Lq * d.M), value, gv))
        return launch_bwd_slab<T>(go, value, shapes, lsi, loc, attn, d, gv, gl, ga, st);
    if constexpr (sizeof(T) == 4) {
        if (knob(MSDA_KNOB_F32_VEC8_BWD) == 1 && LP <= 16 && d.D == 32 &&
            !((reinterpret_cast<uintptr_t>(value) | reinterpret_cast<uintptr_t>(go)) & 31u))
            return launch_bwd<T, 32, 16, 8>(go, value, shapes, lsi, loc, attn, d, gv, gl, ga, st, nullptr, 0);
    }
    switch (d.D) {
        case 16: if constexpr (sizeof(T) == 4) return MSDA_ROUTE_LP(T, 16, launch_bwd)(go, value, shapes, lsi, loc, attn, d, gv, gl, ga, st, nullptr, 0); break;
        case 32: return MSDA_ROUTE_LP(T, 32, launch_bwd)(go, value, shapes, lsi, loc, attn, d, gv, gl, ga, st, nullptr, 0);
        case 64: return MSDA_ROUTE_LP(T, 64, launch_bwd)(go, value, shapes, lsi, loc, attn, d, gv, gl, ga, st, nullptr, 0);
    }
    return cudaErrorInvalidValue;
}

template <typename T, typename TL>
cudaError_t fwd_generic(const T *value, const int64_t *shapes, const int64_t *lsi, const TL *loc, const TL *attn,
                        const Dims &d, T *out, cudaStream_t st) {
    const long long total = (long long)d.N * d.Lq * d.M * d.D;
    long long blocks = (total + 255) / 256;
    const long long cap = (long long)num_sms() * 32;
    if (blocks > cap) blocks = cap;
    msda::msda_fwd_generic<T, TL><<<(int)blocks, 256, 0, st>>>(value, shapes, lsi, loc, attn, d.S, d.M, d.D, d.L, d.Lq,
                                                               d.P, total, out);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}

template <typename T, typename TL, typename GA, bool DET = false>
cudaError_t bwd_generic(const T *go, const T *value, const int64_t *shapes, const int64_t *lsi, const TL *loc,
                        const TL *attn, const Dims &d, GA *gv, TL *gl, TL *ga, cudaStream_t st,
                        unsigned long long *det_acc = nullptr, int det_clog2 = 0) {
    const long long npairs = (long long)d.N * d.Lq * d.M;
    int threads = ((d.D + 31) / 32) * 32;
    if (threads > 256) threads = 256;
    long long blocks = npairs;
    const long long cap = (long long)num_sms() * 64;
    if (blocks > cap) blocks = cap;
    msda::msda_bwd_generic<T, TL, GA, DET><<<(int)blocks, threads, 0, st>>>(go, value, shapes, lsi, loc, attn, d.S, d.M,
                                                                            d.D, d.L, d.Lq, d.P, npairs, gv, gl, ga,
                                                                            det_acc, det_clog2);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}

// ---- deterministic backward (msda_det.cuh) -------------------------------------------------------------------------
// Tiled kernels (linear / TMA / SPLIT, chosen as in the default path) or the generic kernel accumulate into the
// fixed-point sums; the slab / tensor-memory kernels, VEC8 lanes and BF16_FINE_ROWS do not apply.
static_assert(msda::kDetHeaderWords == MSDA_DET_HEADER_WORDS, "accumulator header size");

template <typename T>
cudaError_t bwd_det(const T *go, const T *value, const int64_t *shapes, const int64_t *lsi, const float *loc,
                    const float *attn, const Dims &d, bool aligned, int64_t *acc, float *nf, float *gl, float *ga,
                    float *out32, __nv_bfloat16 *out16, cudaStream_t st) {
    unsigned long long *hdr = reinterpret_cast<unsigned long long *>(acc);
    const long long nval = (long long)d.N * d.S * d.M * d.D;
    int clog2 = 0;                                       // K = Lq * L * P contributions per row at most
    while ((1ll << clog2) < (long long)d.Lq * d.L * d.P) ++clog2;
    cudaError_t err = zero_fill(acc, sizeof(int64_t) * (size_t)(nval + msda::kDetHeaderWords), st);
    if (err != cudaSuccess) return err;
    const int wave = num_sms() * 4;
    msda::msda_det_scale<T><<<wave, 256, 0, st>>>(attn, (long long)d.N * d.Lq * d.M * d.L * d.P, go,
                                                  (long long)d.N * d.Lq * d.M * d.D, hdr);
    msda::msda_det_prepare<<<wave, 256, 0, st>>>(hdr, clog2, nf, nval);
    g_launches.fetch_add(2, std::memory_order_relaxed);
    if ((err = cudaGetLastError()) != cudaSuccess) return err;
    const int LP = d.L * d.P;
    if (aligned && use_fast(sizeof(T), d)) {
        switch (d.D) {
            case 16:
                if constexpr (sizeof(T) == 4) {
                    err = LP <= 16 ? launch_bwd<T, 16, 16, 4, true>(go, value, shapes, lsi, loc, attn, d, nf, gl, ga, st, hdr, clog2)
                                   : launch_bwd<T, 16, 32, 4, true>(go, value, shapes, lsi, loc, attn, d, nf, gl, ga, st, hdr, clog2);
                }
                break;
            case 32:
                err = LP <= 16 ? launch_bwd<T, 32, 16, 4, true>(go, value, shapes, lsi, loc, attn, d, nf, gl, ga, st, hdr, clog2)
                               : launch_bwd<T, 32, 32, 4, true>(go, value, shapes, lsi, loc, attn, d, nf, gl, ga, st, hdr, clog2);
                break;
            case 64:
                err = LP <= 16 ? launch_bwd<T, 64, 16, 4, true>(go, value, shapes, lsi, loc, attn, d, nf, gl, ga, st, hdr, clog2)
                               : launch_bwd<T, 64, 32, 4, true>(go, value, shapes, lsi, loc, attn, d, nf, gl, ga, st, hdr, clog2);
                break;
        }
    } else {
        err = bwd_generic<T, float, float, true>(go, value, shapes, lsi, loc, attn, d, nf, gl, ga, st, hdr, clog2);
    }
    if (err != cudaSuccess) return err;
    long long blocks = (nval + 255) / 256;
    if (blocks > (long long)num_sms() * 16) blocks = (long long)num_sms() * 16;
    msda::msda_det_convert<<<(int)blocks, 256, 0, st>>>(hdr, clog2, nf, nval, out32, out16);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}

}  // namespace

extern "C" {

int msda_abi_version(void) { return MSDA_ABI_VERSION; }

const char *msda_strerror(int code) {
    if (code == 0) return "success";
    if (code == MSDA_E_BADARG) return "msda: bad argument (null pointer, non-positive dimension or unknown knob)";
    if (code == MSDA_E_TOOLARGE) return "msda: problem too large for the kernel index types";
    if (code == MSDA_E_NODEVICE) return "msda: no CUDA device";
    if (code > 0) return cudaGetErrorString(static_cast<cudaError_t>(code));
    return "msda: unknown error";
}

int msda_uses_fast_path(int dtype_bytes, int D, int L, int P) { return fast_ok(dtype_bytes, D, L, P) ? 1 : 0; }

uint64_t msda_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int msda_set_knob(int k, int value) {
    if (k < 0 || k >= MSDA_KNOB_COUNT) return MSDA_E_BADARG;
    Knobs &kn = knobs();
    if (value == MSDA_KNOB_QUERY) return kn.v[k].load(std::memory_order_relaxed);
    const int old = kn.v[k].exchange(value, std::memory_order_relaxed);
    kn.epoch.fetch_add(1, std::memory_order_release);
    return old;
}

// Null pointers are argument errors.  Alignment is a ROUTING property: the tiled / slab kernels need 16-byte aligned
// tensors (vector loads, vector reds); anything else -- e.g. a contiguous view with a storage offset, which the
// reference accepts -- runs on the generic scalar kernels (natural alignment only).
#define MSDA_CHECK_PTRS(ALIGNED, ...)                                    \
    bool ALIGNED = true;                                                 \
    do {                                                                 \
        const void *ptrs_[] = {__VA_ARGS__};                             \
        for (const void *p_ : ptrs_) {                                   \
            if (p_ == nullptr) return MSDA_E_BADARG;                     \
            ALIGNED = ALIGNED && aligned16(p_);                          \
        }                                                                \
    } while (0)

int msda_forward_f32(const float *value, const int64_t *spatial_shapes, const int64_t *level_start_index,
                     const float *sampling_loc, const float *attn_weight, int N, int S, int M, int D, int L, int Lq,
                     int P, float *out, void *stream) {
    const Dims d{N, S, M, D, L, Lq, P};
    if (int e = check_dims(d)) return e;
    MSDA_CHECK_PTRS(al, value, sampling_loc, attn_weight, out);
    if (!spatial_shapes || !level_start_index) return MSDA_E_BADARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (al && use_fast(4, d)) return (int)fwd_fast<float>(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, d, out, st);
    return (int)fwd_generic<float, float>(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, d, out, st);
}

int msda_forward_f64(const double *value, const int64_t *spatial_shapes, const int64_t *level_start_index,
                     const double *sampling_loc, const double *attn_weight, int N, int S, int M, int D, int L, int Lq,
                     int P, double *out, void *stream) {
    const Dims d{N, S, M, D, L, Lq, P};
    if (int e = check_dims(d)) return e;
    if (!value || !spatial_shapes || !level_start_index || !sampling_loc || !attn_weight || !out) return MSDA_E_BADARG;
    return (int)fwd_generic<double, double>(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, d, out,
                                            static_cast<cudaStream_t>(stream));
}

int msda_forward_bf16(const uint16_t *value, const int64_t *spatial_shapes, const int64_t *level_start_index,
                      const float *sampling_loc, const float *attn_weight, int N, int S, int M, int D, int L, int Lq,
                      int P, uint16_t *out, void *stream) {
    const Dims d{N, S, M, D, L, Lq, P};
    if (int e = check_dims(d)) return e;
    MSDA_CHECK_PTRS(al, value, sampling_loc, attn_weight, out);
    if (!spatial_shapes || !level_start_index) return MSDA_E_BADARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const __nv_bfloat16 *v = reinterpret_cast<const __nv_bfloat16 *>(value);
    __nv_bfloat16 *o = reinterpret_cast<__nv_bfloat16 *>(out);
    if (al && use_fast(2, d)) return (int)fwd_fast<__nv_bfloat16>(v, spatial_shapes, level_start_index, sampling_loc, attn_weight, d, o, st);
    return (int)fwd_generic<__nv_bfloat16, float>(v, spatial_shapes, level_start_index, sampling_loc, attn_weight, d, o, st);
}

int msda_backward_f32(const float *grad_out, const float *value, const int64_t *spatial_shapes,
                      const int64_t *level_start_index, const float *sampling_loc, const float *attn_weight, int N,
                      int S, int M, int D, int L, int Lq, int P, float *grad_value, float *grad_sampling_loc,
                      float *grad_attn_weight, void *stream) {
    const Dims d{N, S, M, D, L, Lq, P};
    if (int e = check_dims(d)) return e;
    MSDA_CHECK_PTRS(al, grad_out, value, sampling_loc, attn_weight, grad_value, grad_sampling_loc, grad_attn_weight);
    if (!spatial_shapes || !level_start_index) return MSDA_E_BADARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    bool pdl = false;
    cudaError_t err = zero_fill(grad_value, sizeof(float) * (size_t)N * S * M * D, st, &pdl);
    if (err != cudaSuccess) return (int)err;
    if (al && use_fast(4, d)) {
        t_pdl_next = pdl;
        err = bwd_fast<float>(grad_out, value, spatial_shapes, level_start_index, sampling_loc, attn_weight, d,
                              grad_value, grad_sampling_loc, grad_attn_weight, st);
        t_pdl_next = false;
        return (int)err;
    }
    return (int)bwd_generic<float, float, float>(grad_out, value, spatial_shapes, level_start_index, sampling_loc,
                                                 attn_weight, d, grad_value, grad_sampling_loc, grad_attn_weight, st);
}

int msda_backward_f64(const double *grad_out, const double *value, const int64_t *spatial_shapes,
                      const int64_t *level_start_index, const double *sampling_loc, const double *attn_weight, int N,
                      int S, int M, int D, int L, int Lq, int P, double *grad_value, double *grad_sampling_loc,
                      double *grad_attn_weight, void *stream) {
    const Dims d{N, S, M, D, L, Lq, P};
    if (int e = check_dims(d)) return e;
    if (!grad_out || !value || !spatial_shapes || !level_start_index || !sampling_loc || !attn_weight || !grad_value ||
        !grad_sampling_loc || !grad_attn_weight)
        return MSDA_E_BADARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaError_t err = zero_fill(grad_value, sizeof(double) * (size_t)N * S * M * D, st);
    if (err != cudaSuccess) return (int)err;
    return (int)bwd_generic<double, double, double>(grad_out, value, spatial_shapes, level_start_index, sampling_loc,
                                                    attn_weight, d, grad_value, grad_sampling_loc, grad_attn_weight, st);
}

int msda_backward_bf16(const uint16_t *grad_out, const uint16_t *value, const int64_t *spatial_shapes,
                       const int64_t *level_start_index, const float *sampling_loc, const float *attn_weight, int N,
                       int S, int M, int D, int L, int Lq, int P, float *grad_value_f32, uint16_t *grad_value,
                       float *grad_sampling_loc, float *grad_attn_weight, void *stream) {
    const Dims d{N, S, M, D, L, Lq, P};
    if (int e = check_dims(d)) return e;
    MSDA_CHECK_PTRS(al, grad_out, value, sampling_loc, attn_weight, grad_value_f32, grad_sampling_loc, grad_attn_weight);
    if (!spatial_shapes || !level_start_index) return MSDA_E_BADARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t nval = (size_t)N * S * M * D;
    const __nv_bfloat16 *go = reinterpret_cast<const __nv_bfloat16 *>(grad_out);
    const __nv_bfloat16 *v = reinterpret_cast<const __nv_bfloat16 *>(value);
    const int fine_rows = knob(MSDA_KNOB_BF16_FINE_ROWS);
    if (fine_rows > 0 && grad_value != nullptr && al && use_fast(2, d) && D == 32 && L * P <= 16 &&
        !use_split((unsigned)((long long)N * Lq * M)) && !(reinterpret_cast<uintptr_t>(grad_value) & 15u)) {
        // mixed accumulation: bf16 result zero-filled (fine levels add into it), fp32 scratch zero-filled for the coarse
        // levels only, one rounding pass over the coarse rows at the end -- no full-size fp32 round trip
        __nv_bfloat16 *gv16 = reinterpret_cast<__nv_bfloat16 *>(grad_value);
        cudaError_t e = zero_fill(grad_value, sizeof(uint16_t) * nval, st);
        if (e != cudaSuccess) return (int)e;
        const dim3 hgrid((unsigned)(num_sms() * 2 / (N < 1 ? 1 : N) + 1), (unsigned)N);
        msda::msda_coarse_rows<false><<<hgrid, 256, 0, st>>>(grad_value_f32, gv16, spatial_shapes, level_start_index, L, S,
                                                             M * D, fine_rows);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        e = launch_bwd_mixed(go, v, spatial_shapes, level_start_index, sampling_loc, attn_weight, d, grad_value_f32, gv16,
                             grad_sampling_loc, grad_attn_weight, fine_rows, st);
        if (e != cudaSuccess) return (int)e;
        msda::msda_coarse_rows<true><<<hgrid, 256, 0, st>>>(grad_value_f32, gv16, spatial_shapes, level_start_index, L, S,
                                                            M * D, fine_rows);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        return (int)cudaGetLastError();
    }
    bool pdl = false;
    cudaError_t err = zero_fill(grad_value_f32, sizeof(float) * nval, st, &pdl);
    if (err != cudaSuccess) return (int)err;
    if (al && use_fast(2, d)) {
        t_pdl_next = pdl;
        err = bwd_fast<__nv_bfloat16>(go, v, spatial_shapes, level_start_index, sampling_loc, attn_weight, d,
                                      grad_value_f32, grad_sampling_loc, grad_attn_weight, st);
        t_pdl_next = false;
    } else
        err = bwd_generic<__nv_bfloat16, float, float>(go, v, spatial_shapes, level_start_index, sampling_loc,
                                                       attn_weight, d, grad_value_f32, grad_sampling_loc,
                                                       grad_attn_weight, st);
    if (err != cudaSuccess) return (int)err;
    if (grad_value != nullptr) {
        long long blocks = (long long)((nval + 255) / 256);
        const long long cap = (long long)num_sms() * 16;
        if (blocks > cap) blocks = cap;
        msda::msda_f32_to_bf16<<<(int)blocks, 256, 0, st>>>(grad_value_f32, reinterpret_cast<__nv_bfloat16 *>(grad_value),
                                                            (long long)nval);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        err = cudaGetLastError();
    }
    return (int)err;
}

int msda_backward_det_f32(const float *grad_out, const float *value, const int64_t *spatial_shapes,
                          const int64_t *level_start_index, const float *sampling_loc, const float *attn_weight, int N,
                          int S, int M, int D, int L, int Lq, int P, int64_t *acc, float *grad_value,
                          float *grad_sampling_loc, float *grad_attn_weight, void *stream) {
    const Dims d{N, S, M, D, L, Lq, P};
    if (int e = check_dims(d)) return e;
    MSDA_CHECK_PTRS(al, grad_out, value, sampling_loc, attn_weight, grad_value, grad_sampling_loc, grad_attn_weight);
    if (!spatial_shapes || !level_start_index || !acc || (reinterpret_cast<uintptr_t>(acc) & 7u)) return MSDA_E_BADARG;
    return (int)bwd_det<float>(grad_out, value, spatial_shapes, level_start_index, sampling_loc, attn_weight, d, al, acc,
                               grad_value, grad_sampling_loc, grad_attn_weight, grad_value, nullptr,
                               static_cast<cudaStream_t>(stream));
}

int msda_backward_det_bf16(const uint16_t *grad_out, const uint16_t *value, const int64_t *spatial_shapes,
                           const int64_t *level_start_index, const float *sampling_loc, const float *attn_weight, int N,
                           int S, int M, int D, int L, int Lq, int P, int64_t *acc, float *grad_value_f32,
                           uint16_t *grad_value, float *grad_sampling_loc, float *grad_attn_weight, void *stream) {
    const Dims d{N, S, M, D, L, Lq, P};
    if (int e = check_dims(d)) return e;
    MSDA_CHECK_PTRS(al, grad_out, value, sampling_loc, attn_weight, grad_value_f32, grad_sampling_loc, grad_attn_weight);
    if (!spatial_shapes || !level_start_index || !acc || (reinterpret_cast<uintptr_t>(acc) & 7u)) return MSDA_E_BADARG;
    __nv_bfloat16 *gv16 = reinterpret_cast<__nv_bfloat16 *>(grad_value);
    return (int)bwd_det<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16 *>(grad_out),
                                       reinterpret_cast<const __nv_bfloat16 *>(value), spatial_shapes, level_start_index,
                                       sampling_loc, attn_weight, d, al, acc, grad_value_f32, grad_sampling_loc,
                                       grad_attn_weight, gv16 ? nullptr : grad_value_f32, gv16,
                                       static_cast<cudaStream_t>(stream));
}

}  // extern "C"

// ---- callers of the op --------------------------------------------------------------------------------------------
namespace {
template <int G>
cudaError_t prologue_fwd_launch(const float *proj, const float *ref, const int64_t *shapes, long long npairs, int M, int L,
                                int P, int refdim, float *loc, float *attn, cudaStream_t st) {
    const long long threads = npairs * G;
    msda::msda_prologue_fwd<G><<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(proj, ref, shapes, npairs, M, L, P, refdim, loc, attn);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}
template <int G>
cudaError_t prologue_bwd_launch(const float *gl, const float *ga, const float *attn, const float *ref, const int64_t *shapes,
                                long long npairs, int M, int L, int P, int refdim, float *gp, cudaStream_t st) {
    const long long threads = npairs * G;
    msda::msda_prologue_bwd<G><<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(gl, ga, attn, ref, shapes, npairs, M, L, P, refdim, gp);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}
int group_width(int LP) { return LP <= 4 ? 4 : LP <= 8 ? 8 : LP <= 16 ? 16 : 32; }
}  // namespace

extern "C" {

int msda_prologue_forward_f32(const float *proj, const float *ref, const int64_t *spatial_shapes, int64_t R, int M, int L,
                              int P, int refdim, float *loc, float *attn, void *stream) {
    if (!proj || !ref || !spatial_shapes || !loc || !attn || R <= 0 || M <= 0 || L <= 0 || P <= 0 || L * P > 32 ||
        (refdim != 2 && refdim != 4) || (long long)R * M * 32 >= (1ll << 40))
        return MSDA_E_BADARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long np = (long long)R * M;
    switch (group_width(L * P)) {
        case 4: return (int)prologue_fwd_launch<4>(proj, ref, spatial_shapes, np, M, L, P, refdim, loc, attn, st);
        case 8: return (int)prologue_fwd_launch<8>(proj, ref, spatial_shapes, np, M, L, P, refdim, loc, attn, st);
        case 16: return (int)prologue_fwd_launch<16>(proj, ref, spatial_shapes, np, M, L, P, refdim, loc, attn, st);
        default: return (int)prologue_fwd_launch<32>(proj, ref, spatial_shapes, np, M, L, P, refdim, loc, attn, st);
    }
}

int msda_prologue_backward_f32(const float *grad_loc, const float *grad_attn, const float *attn, const float *ref,
                               const int64_t *spatial_shapes, int64_t R, int M, int L, int P, int refdim,
                               float *grad_proj, void *stream) {
    if (!grad_loc || !grad_attn || !attn || !ref || !spatial_shapes || !grad_proj || R <= 0 || M <= 0 || L <= 0 || P <= 0 ||
        L * P > 32 || (refdim != 2 && refdim != 4))
        return MSDA_E_BADARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long np = (long long)R * M;
    switch (group_width(L * P)) {
        case 4: return (int)prologue_bwd_launch<4>(grad_loc, grad_attn, attn, ref, spatial_shapes, np, M, L, P, refdim, grad_proj, st);
        case 8: return (int)prologue_bwd_launch<8>(grad_loc, grad_attn, attn, ref, spatial_shapes, np, M, L, P, refdim, grad_proj, st);
        case 16: return (int)prologue_bwd_launch<16>(grad_loc, grad_attn, attn, ref, spatial_shapes, np, M, L, P, refdim, grad_proj, st);
        default: return (int)prologue_bwd_launch<32>(grad_loc, grad_attn, attn, ref, spatial_shapes, np, M, L, P, refdim, grad_proj, st);
    }
}

int msda_colsum_f32(const float *x, int64_t rows, int cols, float *out, void *stream) {
    if (!x || !out || rows <= 0 || cols <= 0 || cols % 4 != 0 || !aligned16(x) || !aligned16(out)) return MSDA_E_BADARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaError_t err = cudaMemsetAsync(out, 0, sizeof(float) * (size_t)cols, st);
    if (err != cudaSuccess) return (int)err;
    long long ctas = (long long)num_sms() * 4;
    int rows_per_cta = (int)((rows + ctas - 1) / ctas);
    if (rows_per_cta < 16) rows_per_cta = 16;
    const unsigned grid = (unsigned)((rows + rows_per_cta - 1) / rows_per_cta);
    msda::msda_colsum<<<grid, 256, 0, st>>>(x, rows, cols, rows_per_cta, out);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return (int)cudaGetLastError();
}

int msda_relu_backward_colsum_f32(const float *g, const float *y, int64_t rows, int cols, float *g2, float *colsum, void *stream) {
    if (!g || !y || !g2 || !colsum || rows <= 0 || cols <= 0 || cols % 4 != 0 || !aligned16(g) || !aligned16(y) || !aligned16(g2) ||
        !aligned16(colsum))
        return MSDA_E_BADARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaError_t err = cudaMemsetAsync(colsum, 0, sizeof(float) * (size_t)cols, st);
    if (err != cudaSuccess) return (int)err;
    long long ctas = (long long)num_sms() * 8;
    int rows_per_cta = (int)((rows + ctas - 1) / ctas);
    if (rows_per_cta < 16) rows_per_cta = 16;
    const unsigned grid = (unsigned)((rows + rows_per_cta - 1) / rows_per_cta);
    msda::msda_relu_bwd_colsum<<<grid, 256, 0, st>>>(g, y, rows, cols, rows_per_cta, g2, colsum);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return (int)cudaGetLastError();
}

}  // extern "C"

// ---- deterministic caller reductions: partial rows per CTA in caller scratch, then a fixed-order sum ---------------------
// The grid is a function of (rows, cols) only -- at most kDetParts CTAs -- so the result is bit-identical on any GPU and the
// scratch size is known on the host.
namespace {
constexpr long long kDetParts = 512;
long long det_rows_per_cta(long long rows, int multiple) {
    long long r = (rows + kDetParts - 1) / kDetParts;
    if (r < 16) r = 16;
    return (r + multiple - 1) / multiple * multiple;
}
long long det_parts(long long rows, int multiple) {
    const long long r = det_rows_per_cta(rows, multiple);
    return (rows + r - 1) / r;
}
bool ln_cols_ok(int cols) { return cols == 128 || cols == 256 || cols == 384 || cols == 512; }
cudaError_t sum_partials(const float *part, long long nparts, int cols, float *out, cudaStream_t st) {
    msda::msda_sum_partials<<<(cols + 255) / 256, 256, 0, st>>>(part, (int)nparts, cols, out);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}
}  // namespace

extern "C" {

int msda_colsum_det_scratch_bytes(int64_t rows, int cols, int64_t *bytes) {
    if (!bytes || rows <= 0 || cols <= 0 || cols % 4 != 0) return MSDA_E_BADARG;
    *bytes = (int64_t)(det_parts(rows, 1) * cols * (long long)sizeof(float));
    return 0;
}

int msda_layernorm_backward_det_scratch_bytes(int64_t rows, int cols, int64_t *bytes) {
    if (!bytes || rows <= 0 || !ln_cols_ok(cols)) return MSDA_E_BADARG;
    *bytes = (int64_t)(2 * det_parts(rows, 8) * cols * (long long)sizeof(float));
    return 0;
}

int msda_colsum_det_f32(const float *x, int64_t rows, int cols, float *scratch, float *out, void *stream) {
    if (!x || !out || !scratch || rows <= 0 || cols <= 0 || cols % 4 != 0 || !aligned16(x) || !aligned16(scratch))
        return MSDA_E_BADARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long rpc = det_rows_per_cta(rows, 1), parts = det_parts(rows, 1);
    msda::msda_colsum<true><<<(unsigned)parts, 256, 0, st>>>(x, rows, cols, (int)rpc, scratch);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    const cudaError_t err = cudaGetLastError();
    return (int)(err != cudaSuccess ? err : sum_partials(scratch, parts, cols, out, st));
}

int msda_relu_backward_colsum_det_f32(const float *g, const float *y, int64_t rows, int cols, float *g2, float *scratch,
                                      float *colsum, void *stream) {
    if (!g || !y || !g2 || !scratch || !colsum || rows <= 0 || cols <= 0 || cols % 4 != 0 || !aligned16(g) || !aligned16(y) ||
        !aligned16(g2) || !aligned16(scratch))
        return MSDA_E_BADARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long rpc = det_rows_per_cta(rows, 1), parts = det_parts(rows, 1);
    msda::msda_relu_bwd_colsum<true><<<(unsigned)parts, 256, 0, st>>>(g, y, rows, cols, (int)rpc, g2, scratch);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    const cudaError_t err = cudaGetLastError();
    return (int)(err != cudaSuccess ? err : sum_partials(scratch, parts, cols, colsum, st));
}

int msda_layernorm_backward_det_f32(const float *dy, const float *z, const float *gamma, const float *mean, const float *rstd,
                                    int64_t rows, int cols, float *dz, float *scratch, float *dgamma, float *dbeta,
                                    void *stream) {
    if (!dy || !z || !gamma || !mean || !rstd || !dz || !scratch || !dgamma || !dbeta || rows <= 0 || !ln_cols_ok(cols))
        return MSDA_E_BADARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long rpc = det_rows_per_cta(rows, 8), parts = det_parts(rows, 8);
    float *pg = scratch, *pb = scratch + parts * cols;
    const unsigned grid = (unsigned)parts;
    switch (cols / 128) {
        case 1: msda::msda_layernorm_bwd<1, true><<<grid, 256, 0, st>>>(dy, z, gamma, mean, rstd, rows, (int)rpc, dz, pg, pb); break;
        case 2: msda::msda_layernorm_bwd<2, true><<<grid, 256, 0, st>>>(dy, z, gamma, mean, rstd, rows, (int)rpc, dz, pg, pb); break;
        case 3: msda::msda_layernorm_bwd<3, true><<<grid, 256, 0, st>>>(dy, z, gamma, mean, rstd, rows, (int)rpc, dz, pg, pb); break;
        default: msda::msda_layernorm_bwd<4, true><<<grid, 256, 0, st>>>(dy, z, gamma, mean, rstd, rows, (int)rpc, dz, pg, pb); break;
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t err = cudaGetLastError();
    if (err == cudaSuccess) err = sum_partials(pg, parts, cols, dgamma, st);
    if (err == cudaSuccess) err = sum_partials(pb, parts, cols, dbeta, st);
    return (int)err;
}

int msda_add_layernorm_forward_f32(const float *a, const float *b, const float *gamma, const float *beta, int64_t rows,
                                   int cols, float eps, float *z, float *y, float *mean, float *rstd, void *stream) {
    if (!a || !gamma || !beta || !y || !mean || !rstd || rows <= 0 || (b != nullptr && z == nullptr)) return MSDA_E_BADARG;
    if (cols != 128 && cols != 256 && cols != 384 && cols != 512) return MSDA_E_BADARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const unsigned grid = (unsigned)((rows + 7) / 8);
    switch (cols / 128) {
        case 1: msda::msda_add_layernorm_fwd<1><<<grid, 256, 0, st>>>(a, b, gamma, beta, rows, eps, z, y, mean, rstd); break;
        case 2: msda::msda_add_layernorm_fwd<2><<<grid, 256, 0, st>>>(a, b, gamma, beta, rows, eps, z, y, mean, rstd); break;
        case 3: msda::msda_add_layernorm_fwd<3><<<grid, 256, 0, st>>>(a, b, gamma, beta, rows, eps, z, y, mean, rstd); break;
        default: msda::msda_add_layernorm_fwd<4><<<grid, 256, 0, st>>>(a, b, gamma, beta, rows, eps, z, y, mean, rstd); break;
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return (int)cudaGetLastError();
}

int msda_layernorm_backward_f32(const float *dy, const float *z, const float *gamma, const float *mean, const float *rstd,
                                int64_t rows, int cols, float *dz, float *dgamma, float *dbeta, void *stream) {
    if (!dy || !z || !gamma || !mean || !rstd || !dz || !dgamma || !dbeta || rows <= 0) return MSDA_E_BADARG;
    if (cols != 128 && cols != 256 && cols != 384 && cols != 512) return MSDA_E_BADARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaError_t err = cudaMemsetAsync(dgamma, 0, sizeof(float) * (size_t)cols, st);
    if (err == cudaSuccess) err = cudaMemsetAsync(dbeta, 0, sizeof(float) * (size_t)cols, st);
    if (err != cudaSuccess) return (int)err;
    long long ctas = (long long)num_sms() * 4;
    int rows_per_cta = (int)((rows + ctas - 1) / ctas);
    rows_per_cta = ((rows_per_cta + 7) / 8) * 8;
    const unsigned grid = (unsigned)((rows + rows_per_cta - 1) / rows_per_cta);
    switch (cols / 128) {
        case 1: msda::msda_layernorm_bwd<1><<<grid, 256, 0, st>>>(dy, z, gamma, mean, rstd, rows, rows_per_cta, dz, dgamma, dbeta); break;
        case 2: msda::msda_layernorm_bwd<2><<<grid, 256, 0, st>>>(dy, z, gamma, mean, rstd, rows, rows_per_cta, dz, dgamma, dbeta); break;
        case 3: msda::msda_layernorm_bwd<3><<<grid, 256, 0, st>>>(dy, z, gamma, mean, rstd, rows, rows_per_cta, dz, dgamma, dbeta); break;
        default: msda::msda_layernorm_bwd<4><<<grid, 256, 0, st>>>(dy, z, gamma, mean, rstd, rows, rows_per_cta, dz, dgamma, dbeta); break;
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return (int)cudaGetLastError();
}

}  // extern "C"

// ---- CondInst dynamic mask head -------------------------------------------------------------------------------------
extern "C" {

int msda_condinst_forward_f32(const float *feats, const float *params, const float *refs, const int32_t *inst_start, int N,
                              int H, int W, int I, int max_inst, int stride, int rel_coord, float *logits, void *stream) {
    if (!feats || !params || !refs || !inst_start || !logits || N <= 0 || H <= 0 || W <= 0 || I < 0 || stride <= 0 ||
        max_inst < 0 || (long long)H * W >= (1ll << 30))
        return MSDA_E_BADARG;
    if (I == 0 || max_inst == 0) return 0;
    const int HW = H * W, tile = msda::kCiFwdThreads * msda::kCiFwdPpt;
    const dim3 grid((unsigned)((HW + tile - 1) / tile), (unsigned)((max_inst + msda::kCiChunk - 1) / msda::kCiChunk), (unsigned)N);
    msda::condinst_fwd<<<grid, msda::kCiFwdThreads, 0, static_cast<cudaStream_t>(stream)>>>(feats, params, refs, inst_start, HW,
                                                                                          W, stride, rel_coord, logits);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return (int)cudaGetLastError();
}

int msda_condinst_backward_f32(const float *grad_logits, const float *feats, const float *params, const float *refs,
                               const int32_t *inst_start, int N, int H, int W, int I, int max_inst, int stride, int rel_coord,
                               float *grad_feats, float *grad_params, float *grad_refs, void *stream) {
    if (!grad_logits || !feats || !params || !refs || !inst_start || !grad_feats || !grad_params || !grad_refs || N <= 0 ||
        H <= 0 || W <= 0 || I < 0 || max_inst < 0 || stride <= 0 || (long long)H * W >= (1ll << 30))
        return MSDA_E_BADARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int HW = H * W, tile = msda::kCiThreads * msda::kCiBwdPpt;
    cudaError_t e = cudaMemsetAsync(grad_feats, 0, sizeof(float) * (size_t)N * msda::kCiFeat * HW, st);
    if (e == cudaSuccess && I > 0) e = cudaMemsetAsync(grad_params, 0, sizeof(float) * (size_t)I * msda::kCiParams, st);
    if (e == cudaSuccess && I > 0) e = cudaMemsetAsync(grad_refs, 0, sizeof(float) * (size_t)I * 2, st);
    if (e != cudaSuccess) return (int)e;
    if (I == 0 || max_inst == 0) return 0;
    const dim3 grid((unsigned)((HW + tile - 1) / tile), (unsigned)((max_inst + msda::kCiChunk - 1) / msda::kCiChunk), (unsigned)N);
    msda::condinst_bwd<<<grid, msda::kCiThreads, 0, st>>>(grad_logits, feats, params, refs, inst_start, HW, W, stride, rel_coord,
                                                          grad_feats, grad_params, grad_refs);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return (int)cudaGetLastError();
}

// Partials of the deterministic CondInst backward: [ceil(max_inst / 16)][N][8][H*W] feature partials, then
// [ceil(H*W / 64)][I][171] per-warp sums.
int msda_condinst_backward_det_scratch_bytes(int N, int H, int W, int I, int max_inst, int64_t *bytes) {
    if (!bytes || N <= 0 || H <= 0 || W <= 0 || I < 0 || max_inst < 0 || (long long)H * W >= (1ll << 30)) return MSDA_E_BADARG;
    const long long HW = (long long)H * W, chunks = (max_inst + msda::kCiChunk - 1) / msda::kCiChunk;
    *bytes = (int64_t)(sizeof(float) * (chunks * N * msda::kCiFeat * HW + ((HW + 63) / 64) * (long long)I * msda::kCiSums));
    return 0;
}

int msda_condinst_backward_det_f32(const float *grad_logits, const float *feats, const float *params, const float *refs,
                                   const int32_t *inst_start, int N, int H, int W, int I, int max_inst, int stride,
                                   int rel_coord, float *scratch, float *grad_feats, float *grad_params, float *grad_refs,
                                   void *stream) {
    if (!grad_logits || !feats || !params || !refs || !inst_start || !scratch || !grad_feats || !grad_params || !grad_refs ||
        N <= 0 || H <= 0 || W <= 0 || I < 0 || max_inst < 0 || stride <= 0 || (long long)H * W >= (1ll << 30))
        return MSDA_E_BADARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int HW = H * W, tile = msda::kCiThreads * msda::kCiBwdPpt;
    if (I == 0 || max_inst == 0)
        return (int)cudaMemsetAsync(grad_feats, 0, sizeof(float) * (size_t)N * msda::kCiFeat * HW, st);
    const int chunks = (max_inst + msda::kCiChunk - 1) / msda::kCiChunk;
    float *feat_part = scratch, *sum_part = scratch + (size_t)chunks * N * msda::kCiFeat * HW;
    const dim3 grid((unsigned)((HW + tile - 1) / tile), (unsigned)chunks, (unsigned)N);
    msda::condinst_bwd<true><<<grid, msda::kCiThreads, 0, st>>>(grad_logits, feats, params, refs, inst_start, HW, W, stride,
                                                                rel_coord, grad_feats, grad_params, grad_refs, feat_part,
                                                                sum_part, I);
    const long long total = (long long)N * msda::kCiFeat * HW + (long long)I * msda::kCiSums;
    long long blocks = (total + 255) / 256;
    if (blocks > (long long)num_sms() * 16) blocks = (long long)num_sms() * 16;
    msda::condinst_bwd_reduce<<<(unsigned)blocks, 256, 0, st>>>(feat_part, sum_part, inst_start, N, HW, I, (HW + 63) / 64,
                                                               grad_feats, grad_params, grad_refs);
    g_launches.fetch_add(2, std::memory_order_relaxed);
    return (int)cudaGetLastError();
}

int msda_aligned_bilinear_forward_f32(const float *in, int64_t planes, int h, int w, int factor, float *out, void *stream) {
    if (!in || !out || planes < 0 || planes >= (1ll << 31) || h <= 0 || w <= 0 || factor < 1 ||
        (long long)h * factor * w * factor >= (1ll << 31))
        return MSDA_E_BADARG;
    if (planes == 0) return 0;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const dim3 grid((unsigned)planes, (unsigned)((h * factor + msda::kAbRows - 1) / msda::kAbRows));
    const bool vec = (w * factor) % 4 == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0;
    if (factor == 2 && vec) msda::aligned_bilinear2_fwd<<<grid, 256, 0, st>>>(in, h, w, out);
    else if (vec) msda::aligned_bilinear_fwd<0, 4><<<grid, 256, 0, st>>>(in, h, w, factor, out);
    else msda::aligned_bilinear_fwd<0, 1><<<grid, 256, 0, st>>>(in, h, w, factor, out);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return (int)cudaGetLastError();
}

int msda_aligned_bilinear_backward_f32(const float *grad_out, int64_t planes, int h, int w, int factor, float *grad_in,
                                       void *stream) {
    if (!grad_out || !grad_in || planes < 0 || planes >= (1ll << 31) || h <= 0 || w <= 0 || factor < 1 ||
        (long long)h * factor * w * factor >= (1ll << 31))
        return MSDA_E_BADARG;
    if (planes == 0) return 0;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const dim3 grid((unsigned)planes, (unsigned)((h + msda::kAbRows - 1) / msda::kAbRows));
    const bool vec = w % 2 == 0 && (reinterpret_cast<uintptr_t>(grad_out) & 15) == 0 && (reinterpret_cast<uintptr_t>(grad_in) & 7) == 0;
    if (factor == 2 && vec) msda::aligned_bilinear2_bwd<<<grid, 256, 0, st>>>(grad_out, h, w, grad_in);
    else msda::aligned_bilinear_bwd<0><<<grid, 256, 0, st>>>(grad_out, h, w, factor, grad_in);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return (int)cudaGetLastError();
}

}  // extern "C"

// ---- geometry feeding the op (f-3) --------------------------------------------------------------------------------------
extern "C" {

int msda_valid_counts(const uint8_t *mask, const int64_t *spatial_shapes, const int64_t *level_start_index, int N, int S, int L,
                      int32_t *counts, void *stream) {
    if (!mask || !spatial_shapes || !level_start_index || !counts || N <= 0 || S <= 0 || L <= 0) return MSDA_E_BADARG;
    const int warps = N * L;
    msda::msda_valid_counts<<<(warps * 32 + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(mask, spatial_shapes,
                                                                                                      level_start_index, N, S, L, counts);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return (int)cudaGetLastError();
}

int msda_encoder_ref_points_f32(const float *valid_ratios, const int64_t *spatial_shapes, const int64_t *level_start_index, int N,
                                int S, int L, float *ref, void *stream) {
    if (!valid_ratios || !spatial_shapes || !level_start_index || !ref || N <= 0 || S <= 0 || L <= 0 || !aligned16(ref)) return MSDA_E_BADARG;
    const long long total = (long long)N * S;
    msda::msda_encoder_ref_points<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        valid_ratios, spatial_shapes, level_start_index, N, S, L, ref);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return (int)cudaGetLastError();
}

int msda_encoder_proposals_f32(const uint8_t *mask, const int32_t *counts, const int64_t *spatial_shapes,
                               const int64_t *level_start_index, int N, int S, int L, float base_scale, float *proposals,
                               uint8_t *keep, void *stream) {
    if (!mask || !counts || !spatial_shapes || !level_start_index || !proposals || !keep || N <= 0 || S <= 0 || L <= 0 || L > 30 ||
        !aligned16(proposals))
        return MSDA_E_BADARG;
    const long long total = (long long)N * S;
    msda::msda_encoder_proposals<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        mask, counts, spatial_shapes, level_start_index, N, S, L, base_scale, proposals, keep);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return (int)cudaGetLastError();
}

int msda_sine_pos_embed_forward_f32(const float *pos, int64_t R, int n, int F, float temperature, int exchange_xy, float *out,
                                    void *stream) {
    if (!pos || !out || R <= 0 || n <= 0 || F <= 0) return MSDA_E_BADARG;
    const long long warps = (long long)R * n;
    msda::msda_sine_pos_embed<false><<<(unsigned)((warps * 32 + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        pos, nullptr, R, n, F, temperature, exchange_xy, out);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return (int)cudaGetLastError();
}

int msda_sine_pos_embed_backward_f32(const float *pos, const float *grad_out, int64_t R, int n, int F, float temperature,
                                     int exchange_xy, float *grad_pos, void *stream) {
    if (!pos || !grad_out || !grad_pos || R <= 0 || n <= 0 || F <= 0) return MSDA_E_BADARG;
    const long long warps = (long long)R * n;
    msda::msda_sine_pos_embed<true><<<(unsigned)((warps * 32 + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        pos, grad_out, R, n, F, temperature, exchange_xy, grad_pos);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return (int)cudaGetLastError();
}

}  // extern "C"
