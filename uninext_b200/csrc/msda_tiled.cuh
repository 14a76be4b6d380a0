// msda_tiled.cuh -- the sm_100a fast path: persistent, row-vectorised gather kernels (forward and backward).
//
// Thread mapping.  A value row of one head is D contiguous elements; LPR = D / kElems lanes cover it with one 16-byte
// access each (fp32 D=32: 8 lanes, bf16 D=32: 4 lanes).  A warp therefore carries GPW = 32 / LPR "groups"; each group
// owns one (batch, query, head) pair at a time.  Work inside a group is split two ways:
//   stage 1 (by tap):     lane `sub` resolves taps sub, sub+LPR, ... : reads (x, y, a), resolves the bilinear
//                         geometry once (tap_geometry) and publishes a 24-byte tap record {4 masked corner weights,
//                         2 clamped row indices} to a per-warp shared-memory slab (conflict-free layout).
//   stage 2 (by channel): for every tap each lane reads the record (one LDS.128 + one LDS.64, broadcast inside the
//                         group) and issues four 16-byte row loads for ITS channel slice.
// This removes the reference forward kernel's 32x-redundant per-channel index arithmetic and scalar loads
// (cuh:272-296) and the reference backward kernel's per-tap __syncthreads + serial shared-memory reductions
// (cuh:347-401): the backward channel reduction is a shuffle reduce-scatter that leaves tap j's sums on lane j,
// i.e. on the lane that already holds that tap's geometry.
//
// Work decomposition.  The grid is persistent (SM count x resident CTAs); CTA c walks tiles c, c+G, c+2G, ...
// Two slot orders:
//   linear  -- a tile is one CTA iteration of consecutive pairs in memory order (the default);
//   patches -- used when Lq == S and the level table tiles [0, S) exactly, i.e. queries ARE the pixels of the pyramid
//              (encoder self-attention, deformable_transformer.py:280-292): a tile is one head of an 8x8 pixel patch,
//              so the rows gathered by neighbouring queries of the same head overlap in L1 while the tile is resident.
//              Purely a scheduling choice: every pair is still processed exactly once, results do not depend on it.
//              Off by default (MSDA_PATCHES=1): it raises the L1 hit rate but the kernels are not L1-miss bound.
// Template switches: TMA   -- stage 1 reads (x, y, a) from a per-warp double buffer filled one iteration ahead by
//                             cp.async.bulk + mbarrier (linear order only; default on);
//                    SPLIT -- small launches: the groups of a warp share one pair and split its taps (see kernel body).
#pragma once

#include "msda_common.cuh"
#include "msda_det.cuh"

namespace msda {

constexpr int kTiledThreads = 256;
constexpr int kTiledWarps = kTiledThreads / 32;
constexpr int kPatch = 8;                       // pixel patch edge (patches mode)
constexpr int kTileSlots = kPatch * kPatch;     // (pair) slots per tile, both modes

struct WorkMap {
    int H[kMaxLevels], W[kMaxLevels], start[kMaxLevels];
    int pcols[kMaxLevels];           // patches per patch-row of level l
    int pfirst[kMaxLevels + 1];      // first patch index of level l within one batch element
    int patches;                     // 1 when the patch order is in use
    unsigned ntiles;
    unsigned linear_tile;            // pairs per tile in linear order (= one CTA iteration)
};

// Every CTA derives the same map from the (device-resident) level table: no host read of spatial_shapes is needed.
__device__ __forceinline__ void build_work_map(WorkMap &wm, const int64_t *shapes, const int64_t *lsi, int L, int N,
                                               int S, int Lq, int M, unsigned npairs, int allow_patches,
                                               unsigned linear_tile) {
    if (threadIdx.x == 0) {
        int run = 0, np = 0;
        bool tiled = (Lq == S) && allow_patches;
        for (int l = 0; l < L; ++l) {
            const int h = (int)shapes[2 * l], w = (int)shapes[2 * l + 1], st = (int)lsi[l];
            wm.H[l] = h; wm.W[l] = w; wm.start[l] = st;
            tiled = tiled && (st == run) && h > 0 && w > 0;
            run += h * w;
            wm.pcols[l] = (w + kPatch - 1) / kPatch;
            wm.pfirst[l] = np;
            np += wm.pcols[l] * ((h + kPatch - 1) / kPatch);
        }
        wm.pfirst[L] = np;
        tiled = tiled && (run == S);
        wm.patches = tiled ? 1 : 0;
        wm.ntiles = tiled ? (unsigned)N * (unsigned)M * (unsigned)np : (npairs + linear_tile - 1) / linear_tile;
        wm.linear_tile = linear_tile;
    }
    __syncthreads();
}

struct TileCtx {          // CTA-uniform description of the current tile
    int b, m, H, W, start, py0, px0;
    unsigned base_pair;
};

__device__ __forceinline__ TileCtx decode_tile(const WorkMap &wm, unsigned tile, int L, int M) {
    TileCtx t;
    if (wm.patches) {
        t.m = (int)(tile % (unsigned)M);               // heads fastest: the 8 tiles of a patch run at about the same
        unsigned r = tile / (unsigned)M;               // time and share DRAM pages of loc / attn / out
        const unsigned per_b = (unsigned)wm.pfirst[L];
        t.b = (int)(r / per_b);
        int p = (int)(r % per_b);
        int l = 0;
        while (l + 1 < L && p >= wm.pfirst[l + 1]) ++l;
        p -= wm.pfirst[l];
        t.H = wm.H[l]; t.W = wm.W[l]; t.start = wm.start[l];
        t.py0 = (p / wm.pcols[l]) * kPatch;
        t.px0 = (p % wm.pcols[l]) * kPatch;
        t.base_pair = 0;
    } else {
        t.b = t.m = t.H = t.W = t.start = t.py0 = t.px0 = 0;
        t.base_pair = tile * wm.linear_tile;
    }
    return t;
}

// Which (b, q, m) pair does this group handle in iteration `it` of the tile?  Returns false for idle slots.
// PPW = pairs per warp: GPW (one pair per group) or 1 (SPLIT: the groups of a warp share one pair and split its taps).
template <int GPW, int PPW>
__device__ __forceinline__ bool slot_pair(const WorkMap &wm, const TileCtx &t, int it, int warp, int grp, int Lq, int M,
                                          unsigned npairs, unsigned &pair, int &b, int &m) {
    if (wm.patches) {
        const int y = t.py0 + warp, x = t.px0 + it * GPW + grp;       // warp = patch row, groups = neighbours in x
        const bool ok = (y < t.H) && (x < t.W);
        const int q = ok ? t.start + y * t.W + x : t.start;
        b = t.b; m = t.m;
        pair = ((unsigned)t.b * (unsigned)Lq + (unsigned)q) * (unsigned)M + (unsigned)t.m;
        return ok;
    }
    const unsigned p = t.base_pair + (unsigned)(warp * PPW + (PPW == 1 ? 0 : grp));     // linear tiles: a single iteration
    const bool ok = p < npairs;
    pair = ok ? p : npairs - 1;
    m = (int)(pair % (unsigned)M);
    b = (int)((pair / (unsigned)M) / (unsigned)Lq);
    return ok;
}

// Per-warp slab for tap records.  Strides are padded so that (a) the LPR records of a group are contiguous (one
// wavefront per quarter-warp store) and (b) the GPW concurrent broadcast reads fall into disjoint banks.
template <int LPR>
struct TapSlab {
    static constexpr int GPW = 32 / LPR;
    static constexpr int kStrideW = LPR * 16 + 16;     // bytes between groups, weight records (float4)
    static constexpr int kStrideR = LPR * 8 + 8;       // bytes between groups, row records (int2)
    static constexpr int kBytes = GPW * (kStrideW + kStrideR);
    unsigned char *w, *r;
    __device__ __forceinline__ TapSlab(unsigned char *warp_base, int grp)
        : w(warp_base + grp * kStrideW), r(warp_base + GPW * kStrideW + grp * kStrideR) {}
    __device__ __forceinline__ void put(int j, float4 wt, int2 rows) {
        *reinterpret_cast<float4 *>(w + j * 16) = wt;
        *reinterpret_cast<int2 *>(r + j * 8) = rows;
    }
    __device__ __forceinline__ float4 weights(int j) const { return *reinterpret_cast<const float4 *>(w + j * 16); }
    __device__ __forceinline__ int2 rows(int j) const { return *reinterpret_cast<const int2 *>(r + j * 8); }
};


// ---- TMA (bulk async copy) staging of one warp-iteration's sampling locations and attention weights -----------------
// Linear order only: the GPW pairs a warp handles in one iteration are consecutive in memory, so their taps are two
// contiguous runs (GPW*LP*8 bytes of (x,y), GPW*LP*4 bytes of weights).  Lane 0 issues the two cp.async.bulk copies for
// the NEXT iteration into the other stage of a per-warp double buffer and the warp waits on that stage's mbarrier when
// it gets there: the taps arrive without occupying registers or issue slots, one iteration ahead of their use.
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

template <int GPW, int LP_MAX, bool ENABLED>
struct TapStage {                       // per-warp double buffer
    static constexpr int kLoc = GPW * LP_MAX * 8, kAttn = GPW * LP_MAX * 4;
    static constexpr int kBytes = ENABLED ? 2 * (kLoc + kAttn) : 16;
};

// ------------------------------------------------------------------------------------------------------------
// forward:  out[b,q,m,:] = sum_taps a * bilinear(value_l[b,:,m,:], x, y)            (reference cuh:237-299)
// ------------------------------------------------------------------------------------------------------------
// PACKED (bf16 storage, VEC = 8 only): the four corners of a tap are blended in packed bf16 (one HMUL2 + three HFMA2 per
// 2 channels, corner weights broadcast as bf16x2 in the tap record) and only the blended tap is widened and accumulated in
// fp32 -- 4 packed ops + 2 widen + 2 adds per word instead of 8 widen + 8 FFMA.  The bf16 forward is issue-bound on exactly
// that unpack / FFMA stream (smsp__issue_active 68 %, profiles/r01k_enc_bf16_ncu.md).  Costs ~3 bf16 roundings per tap.
template <typename T, int VEC, int D, int LP_MAX, int MIN_CTAS, bool TMA, bool SPLIT, bool PACKED = false>
__global__ void __launch_bounds__(kTiledThreads, MIN_CTAS)
msda_fwd_tiled(const T *__restrict__ value, const int64_t *__restrict__ shapes, const int64_t *__restrict__ lsi,
               const float *__restrict__ loc, const float *__restrict__ attn,
               int N, int S, int M, int L, int Lq, int P, unsigned npairs, int allow_patches, T *__restrict__ out)
{
    constexpr int LPR = D / VEC;            // lanes per row
    constexpr int GPW = 32 / LPR;           // groups per warp
    // SPLIT (small problems, e.g. decoder-style calls): the GPW groups of a warp share ONE pair and take LP_MAX/GPW taps
    // each, so a pair's 4*L*P row loads are spread over the whole warp instead of queuing behind one group -- 4x more
    // loads in flight per pair when the launch is too small to hide latency with other warps.
    constexpr int PPW = SPLIT ? 1 : GPW;                    // pairs in flight per warp
    constexpr int TPG = SPLIT ? LP_MAX / GPW : LPR;         // live tap records per group and round
    constexpr int NSL = SPLIT ? 1 : LP_MAX / LPR;           // record rounds
    constexpr int ITERS = SPLIT ? 1 : kTileSlots / (kTiledWarps * GPW);
    static_assert(D % VEC == 0 && (LPR & (LPR - 1)) == 0 && LPR <= 32 && LP_MAX % LPR == 0, "bad tiling");
    static_assert(SPLIT || (kTileSlots % (kTiledWarps * GPW) == 0 && ITERS >= 1), "tile must be whole iterations");
    static_assert(!SPLIT || (LP_MAX % GPW == 0 && LP_MAX / GPW <= LPR && !TMA), "SPLIT: one record round, LDG taps");
    static_assert(!PACKED || (sizeof(T) == 2 && VEC == 8), "PACKED blends bf16 rows, 8 channels (one 16-byte load) per lane");

    __shared__ WorkMap wm;
    __shared__ __align__(16) unsigned char slab_mem[kTiledWarps * TapSlab<LPR>::kBytes];
    build_work_map(wm, shapes, lsi, L, N, S, Lq, M, npairs, SPLIT ? 0 : allow_patches, kTiledWarps * PPW);

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sub = lane % LPR, grp = lane / LPR;
    const int LP = L * P;
    const unsigned row_bytes = (unsigned)(M * D) * (unsigned)sizeof(T);
    TapSlab<LPR> slab(slab_mem + warp * TapSlab<LPR>::kBytes, grp);

    // per-warp TMA double buffer for (x, y, a) -- linear order only (the host passes TMA=true only then)
    using Stage = TapStage<GPW, LP_MAX, TMA>;
    __shared__ __align__(128) unsigned char stage_mem[kTiledWarps * Stage::kBytes];
    __shared__ __align__(8) unsigned long long stage_bar[kTiledWarps * 2];
    unsigned char *my_stage = stage_mem + warp * Stage::kBytes;
    unsigned long long *my_bar = stage_bar + warp * 2;
    unsigned tma_iter = 0;
    auto stage_issue = [&](unsigned tile, unsigned st) {          // lane 0: taps of this warp's slots in `tile` -> stage st
        const unsigned first = tile * wm.linear_tile + (unsigned)(warp * GPW);
        if (first < npairs) {
            const unsigned n = min((unsigned)GPW, npairs - first);
            const unsigned lb = n * (unsigned)LP * 8u, ab = n * (unsigned)LP * 4u;
            unsigned char *dst = my_stage + st * (Stage::kLoc + Stage::kAttn);
            mbar_expect_tx(my_bar + st, lb + ab);
            bulk_g2s(dst, loc + (size_t)first * LP * 2, lb, my_bar + st);
            bulk_g2s(dst + Stage::kLoc, attn + (size_t)first * LP, ab, my_bar + st);
        }
    };
    if constexpr (TMA) {
        if (lane == 0) {
            mbar_init(my_bar, 1); mbar_init(my_bar + 1, 1);
            mbar_fence_init();
            if (blockIdx.x < wm.ntiles) stage_issue(blockIdx.x, 0);
        }
        __syncwarp();
    }

    for (unsigned tile = blockIdx.x; tile < wm.ntiles; tile += gridDim.x) {
        const TileCtx tc = decode_tile(wm, tile, L, M);
        const int iters = wm.patches ? ITERS : 1;
#pragma unroll 1
        for (int it = 0; it < iters; ++it) {
            unsigned pair; int b, m;
            const bool active = slot_pair<GPW, PPW>(wm, tc, it, warp, grp, Lq, M, npairs, pair, b, m);
            const float2 *st_loc = nullptr; const float *st_attn = nullptr;
            if constexpr (TMA) {
                const unsigned st = tma_iter & 1u;
                __syncwarp();                                  // everyone is done with the stage about to be refilled
                if (lane == 0 && tile + gridDim.x < wm.ntiles) stage_issue(tile + gridDim.x, st ^ 1u);
                if (tile * wm.linear_tile + (unsigned)(warp * GPW) < npairs) mbar_wait(my_bar + st, (tma_iter >> 1) & 1u);
                const unsigned char *src = my_stage + st * (Stage::kLoc + Stage::kAttn);
                st_loc = reinterpret_cast<const float2 *>(src) + grp * LP;
                st_attn = reinterpret_cast<const float *>(src + Stage::kLoc) + grp * LP;
                ++tma_iter;
            }

            // ---- stage 1: this lane resolves its taps (dead taps: zero weight, row 0) ----
            float4 tw[NSL];
            int2 tr[NSL];
#pragma unroll
            for (int k = 0; k < NSL; ++k) {
                const int s = SPLIT ? grp * TPG + sub : sub + k * LPR;
                tw[k] = make_float4(0.f, 0.f, 0.f, 0.f);
                tr[k] = make_int2(0, 0);
                if ((!SPLIT || sub < TPG) && s < LP && active) {
                    const size_t t = (size_t)pair * LP + s;
                    const float2 xy = TMA ? st_loc[s] : __ldg(reinterpret_cast<const float2 *>(loc) + t);
                    const float a = TMA ? st_attn[s] : __ldg(attn + t);
                    const int l = s / P;
                    const TapGeom g = tap_geometry(xy.x, xy.y, wm.H[l], wm.W[l], wm.start[l]);
                    tw[k] = masked_weights(g, a);
                    if constexpr (PACKED) {            // record carries each corner weight as a broadcast bf16x2 pattern
                        const __nv_bfloat162 a2 = __floats2bfloat162_rn(tw[k].x, tw[k].x), b2 = __floats2bfloat162_rn(tw[k].y, tw[k].y),
                                             c2 = __floats2bfloat162_rn(tw[k].z, tw[k].z), d2 = __floats2bfloat162_rn(tw[k].w, tw[k].w);
                        tw[k] = make_float4(__uint_as_float(*reinterpret_cast<const unsigned *>(&a2)),
                                            __uint_as_float(*reinterpret_cast<const unsigned *>(&b2)),
                                            __uint_as_float(*reinterpret_cast<const unsigned *>(&c2)),
                                            __uint_as_float(*reinterpret_cast<const unsigned *>(&d2)));
                    }
                    tr[k] = make_int2(g.r0, g.r1 | (g.dw << 31));
                }
            }

            // ---- stage 2: gather rows for this lane's channel slice ----
            const unsigned char *base = reinterpret_cast<const unsigned char *>(
                value + ((size_t)b * S * M + m) * D + (size_t)sub * VEC);
            float acc[VEC];
#pragma unroll
            for (int e = 0; e < VEC; ++e) acc[e] = 0.f;
#pragma unroll
            for (int k = 0; k < NSL; ++k) {
                __syncwarp();                      // previous records fully consumed
                slab.put(sub, tw[k], tr[k]);
                __syncwarp();
#pragma unroll
                for (int j = 0; j < TPG; ++j) {
                    const float4 w = slab.weights(j);
                    const int2 rr = slab.rows(j);
                    const unsigned dwo = (rr.y < 0) ? row_bytes : 0u;
                    const unsigned char *p0 = base + (unsigned long long)(unsigned)rr.x * row_bytes;
                    const unsigned char *p1 = base + (unsigned long long)(unsigned)(rr.y & 0x7fffffff) * row_bytes;
                    if constexpr (PACKED) {
                        const uint4 q00 = __ldg(reinterpret_cast<const uint4 *>(p0)), q01 = __ldg(reinterpret_cast<const uint4 *>(p0 + dwo));
                        const uint4 q10 = __ldg(reinterpret_cast<const uint4 *>(p1)), q11 = __ldg(reinterpret_cast<const uint4 *>(p1 + dwo));
                        const unsigned u00[4] = {q00.x, q00.y, q00.z, q00.w}, u01[4] = {q01.x, q01.y, q01.z, q01.w};
                        const unsigned u10[4] = {q10.x, q10.y, q10.z, q10.w}, u11[4] = {q11.x, q11.y, q11.z, q11.w};
                        const unsigned wx = __float_as_uint(w.x), wy = __float_as_uint(w.y), wz = __float_as_uint(w.z),
                                       ww = __float_as_uint(w.w);
                        auto b2 = [](unsigned u) { return *reinterpret_cast<const __nv_bfloat162 *>(&u); };
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            __nv_bfloat162 t = __hmul2(b2(wx), b2(u00[i]));
                            t = __hfma2(b2(wy), b2(u01[i]), t);
                            t = __hfma2(b2(wz), b2(u10[i]), t);
                            t = __hfma2(b2(ww), b2(u11[i]), t);
                            const unsigned tu = *reinterpret_cast<const unsigned *>(&t);
                            acc[2 * i] += __uint_as_float(tu << 16);
                            acc[2 * i + 1] += __uint_as_float(tu & 0xffff0000u);
                        }
                    } else {
                    float v00[VEC], v01[VEC], v10[VEC], v11[VEC];
                    RowVec<T, VEC>::load(reinterpret_cast<const T *>(p0), v00);
                    RowVec<T, VEC>::load(reinterpret_cast<const T *>(p0 + dwo), v01);
                    RowVec<T, VEC>::load(reinterpret_cast<const T *>(p1), v10);
                    RowVec<T, VEC>::load(reinterpret_cast<const T *>(p1 + dwo), v11);
#pragma unroll
                    for (int e = 0; e < VEC; ++e) {
                        acc[e] = fmaf(w.x, v00[e], acc[e]);
                        acc[e] = fmaf(w.y, v01[e], acc[e]);
                        acc[e] = fmaf(w.z, v10[e], acc[e]);
                        acc[e] = fmaf(w.w, v11[e], acc[e]);
                    }
                    }
                }
            }
            if constexpr (SPLIT) {                  // the groups hold partial sums over disjoint taps of the same pair
#pragma unroll
                for (int d = LPR; d < 32; d <<= 1) {
#pragma unroll
                    for (int e = 0; e < VEC; ++e) acc[e] += __shfl_xor_sync(kFullMask, acc[e], d);
                }
            }
            if (active && (!SPLIT || grp == 0)) RowVec<T, VEC>::store(out + (size_t)pair * D + (size_t)sub * VEC, acc);
        }
    }
}

// Shuffle reduce-scatter inside a group of LPR lanes: on entry part[j][c] is this lane's partial sum for tap j,
// corner c; on exit res[c] is the full group sum for tap `sub`.  log2(LPR) rounds, 4*LPR/2^r shuffles in round r.
template <int LPR>
__device__ __forceinline__ void group_reduce_scatter(float (&part)[LPR][4], int sub, float (&res)[4]) {
#pragma unroll
    for (int d = LPR / 2; d >= 1; d /= 2) {
        const bool upper = (sub & d) != 0;
#pragma unroll
        for (int j = 0; j < d; ++j) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const float lo = part[j][c], hi = part[j + d][c];
                const float send = upper ? lo : hi;
                const float keep = upper ? hi : lo;
                part[j][c] = keep + __shfl_xor_sync(kFullMask, send, d);
            }
        }
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) res[c] = part[0][c];
}

// ------------------------------------------------------------------------------------------------------------
// backward (reference cuh:87-159 + cuh:301-403):
//   grad_value[corner rows] += w_corner * a * g            (16-byte vector reductions, fp32 accumulator)
//   grad_attn[tap]  = sum_c g[c] * val[c]
//   grad_loc[tap].x = W_l * a * sum_c g[c] * gw[c] ;  .y = H_l * a * sum_c g[c] * gh[c]
// Per tap only the four corner dot products  dot_k = sum_c g[c] * V_k[c]  cross lanes; the bilinear coefficients are
// applied afterwards by the single lane that owns the tap.
// ------------------------------------------------------------------------------------------------------------
// MIXED (bf16 storage only): grad_value of the FINE levels (H_l * W_l >= fine_min_rows: the big maps, whose rows
// collect a few dozen contributions each) is accumulated directly in the bf16 output with packed 8-byte reds -- half the
// bytes through the SM's crossbar port, which is what bounds this kernel -- while the coarse levels (hundreds to
// thousands of contributions per row) keep the fp32 accumulator.  The fine flag travels in bit 31 of the record's row
// index (rows are < 2^30).
// DET (msda_det.cuh): grad_value is accumulated as 64-bit fixed point in det_acc (header, then the sums), with the
// same taps, skip rule and fp32 products (det_contrib) as msda_bwd_generic<DET>; grad_value itself only receives
// non-finite contributions.  u64 reds have no vector form, so each group first transposes its output gradient: in
// red k lane `sub` owns channel k * LPR + sub, and the LPR lanes of a group write LPR consecutive words of one row.
template <typename T, int VEC, int D, int LP_MAX, int MIN_CTAS, bool TMA, bool SPLIT, bool MIXED = false, bool DET = false>
__global__ void __launch_bounds__(kTiledThreads, MIN_CTAS)
msda_bwd_tiled(const T *__restrict__ grad_out, const T *__restrict__ value,
               const int64_t *__restrict__ shapes, const int64_t *__restrict__ lsi,
               const float *__restrict__ loc, const float *__restrict__ attn,
               int N, int S, int M, int L, int Lq, int P, unsigned npairs, int allow_patches,
               float *__restrict__ grad_value, float *__restrict__ grad_loc, float *__restrict__ grad_attn,
               __nv_bfloat16 *__restrict__ grad_value_bf16, int fine_min_rows, unsigned long long *__restrict__ det_acc,
               int det_clog2)
{
    static_assert(!MIXED || (sizeof(T) == 2 && VEC == 4), "MIXED accumulates bf16 rows with 8-byte packed reds");
    static_assert(!DET || (!MIXED && VEC == 4), "DET: fp32 contributions, 4 channels per lane");
    constexpr int LPR = D / VEC;
    constexpr int GPW = 32 / LPR;
    constexpr int PPW = SPLIT ? 1 : GPW;                    // see msda_fwd_tiled
    constexpr int TPG = SPLIT ? LP_MAX / GPW : LPR;
    constexpr int NSL = SPLIT ? 1 : LP_MAX / LPR;
    constexpr int ITERS = SPLIT ? 1 : kTileSlots / (kTiledWarps * GPW);
    static_assert(D % VEC == 0 && (LPR & (LPR - 1)) == 0 && LPR <= 32 && LP_MAX % LPR == 0, "bad tiling");
    static_assert(!SPLIT || (LP_MAX % GPW == 0 && LP_MAX / GPW <= LPR && !TMA), "SPLIT: one record round, LDG taps");

    __shared__ WorkMap wm;
    __shared__ __align__(16) unsigned char slab_mem[kTiledWarps * TapSlab<LPR>::kBytes];
    build_work_map(wm, shapes, lsi, L, N, S, Lq, M, npairs, SPLIT ? 0 : allow_patches, kTiledWarps * PPW);

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sub = lane % LPR, grp = lane / LPR;
    const int LP = L * P;
    const unsigned row_elems = (unsigned)(M * D);
    TapSlab<LPR> slab(slab_mem + warp * TapSlab<LPR>::kBytes, grp);

    // per-warp TMA double buffer for (x, y, a) -- linear order only (the host passes TMA=true only then)
    using Stage = TapStage<GPW, LP_MAX, TMA>;
    __shared__ __align__(128) unsigned char stage_mem[kTiledWarps * Stage::kBytes];
    __shared__ __align__(8) unsigned long long stage_bar[kTiledWarps * 2];
    unsigned char *my_stage = stage_mem + warp * Stage::kBytes;
    unsigned long long *my_bar = stage_bar + warp * 2;
    unsigned tma_iter = 0;
    auto stage_issue = [&](unsigned tile, unsigned st) {          // lane 0: taps of this warp's slots in `tile` -> stage st
        const unsigned first = tile * wm.linear_tile + (unsigned)(warp * GPW);
        if (first < npairs) {
            const unsigned n = min((unsigned)GPW, npairs - first);
            const unsigned lb = n * (unsigned)LP * 8u, ab = n * (unsigned)LP * 4u;
            unsigned char *dst = my_stage + st * (Stage::kLoc + Stage::kAttn);
            mbar_expect_tx(my_bar + st, lb + ab);
            bulk_g2s(dst, loc + (size_t)first * LP * 2, lb, my_bar + st);
            bulk_g2s(dst + Stage::kLoc, attn + (size_t)first * LP, ab, my_bar + st);
        }
    };
    if constexpr (TMA) {
        if (lane == 0) {
            mbar_init(my_bar, 1); mbar_init(my_bar + 1, 1);
            mbar_fence_init();
            if (blockIdx.x < wm.ntiles) stage_issue(blockIdx.x, 0);
        }
        __syncwarp();
    }
    pdl_wait_primary();      // grad_value's zero-fill (msda_zero_fill as PDL primary) is complete and visible from here on
    DetScale ds{};
    if constexpr (DET) ds = det_scale(det_acc, det_clog2);

    for (unsigned tile = blockIdx.x; tile < wm.ntiles; tile += gridDim.x) {
        const TileCtx tc = decode_tile(wm, tile, L, M);
        const int iters = wm.patches ? ITERS : 1;
#pragma unroll 1
        for (int it = 0; it < iters; ++it) {
            unsigned pair; int b, m;
            const bool active = slot_pair<GPW, PPW>(wm, tc, it, warp, grp, Lq, M, npairs, pair, b, m);
            const float2 *st_loc = nullptr; const float *st_attn = nullptr;
            if constexpr (TMA) {
                const unsigned st = tma_iter & 1u;
                __syncwarp();                                  // everyone is done with the stage about to be refilled
                if (lane == 0 && tile + gridDim.x < wm.ntiles) stage_issue(tile + gridDim.x, st ^ 1u);
                if (tile * wm.linear_tile + (unsigned)(warp * GPW) < npairs) mbar_wait(my_bar + st, (tma_iter >> 1) & 1u);
                const unsigned char *src = my_stage + st * (Stage::kLoc + Stage::kAttn);
                st_loc = reinterpret_cast<const float2 *>(src) + grp * LP;
                st_attn = reinterpret_cast<const float *>(src + Stage::kLoc) + grp * LP;
                ++tma_iter;
            }

            float g[VEC];
            RowVec<T, VEC>::load(grad_out + (size_t)pair * D + (size_t)sub * VEC, g);
            float gt[VEC];                       // DET: gt[k] = g of channel k * LPR + sub
            if constexpr (DET) {
#pragma unroll
                for (int k = 0; k < VEC; ++k) {
                    const int ch = k * LPR + sub;
                    gt[k] = 0.f;
#pragma unroll
                    for (int e = 0; e < VEC; ++e) {
                        const float t = __shfl_sync(kFullMask, g[e], ch / VEC, LPR);
                        if (e == ch % VEC) gt[k] = t;
                    }
                }
            }

            // ---- stage 1 ----
            float4 tw[NSL];
            int2 tr[NSL];
            float tlh[NSL], tlw[NSL], ta[NSL];
            unsigned tmeta[NSL];                 // corner mask | level << 4
#pragma unroll
            for (int k = 0; k < NSL; ++k) {
                const int s = SPLIT ? grp * TPG + sub : sub + k * LPR;
                tw[k] = make_float4(0.f, 0.f, 0.f, 0.f);
                tr[k] = make_int2(0, 0);
                tlh[k] = tlw[k] = ta[k] = 0.f; tmeta[k] = 0;
                if ((!SPLIT || sub < TPG) && s < LP && active) {
                    const size_t t = (size_t)pair * LP + s;
                    const float2 xy = TMA ? st_loc[s] : __ldg(reinterpret_cast<const float2 *>(loc) + t);
                    const float a = TMA ? st_attn[s] : __ldg(attn + t);
                    const int l = s / P;
                    const TapGeom gm = tap_geometry(xy.x, xy.y, wm.H[l], wm.W[l], wm.start[l]);
                    tw[k] = masked_weights(gm, a);
                    const int fine = (MIXED && wm.H[l] * wm.W[l] >= fine_min_rows) ? (int)0x80000000 : 0;
                    tr[k] = make_int2(gm.r0 | fine, gm.r1 | (gm.dw << 31));
                    tlh[k] = gm.lh; tlw[k] = gm.lw; ta[k] = a; tmeta[k] = gm.mask | ((unsigned)l << 4);
                }
            }

            const size_t slab_off = ((size_t)b * S * M + m) * D + (size_t)sub * VEC;
            const T *base = value + slab_off;
            float *gbase = grad_value + slab_off;

            // ---- stage 2 ----
#pragma unroll
            for (int k = 0; k < NSL; ++k) {
                __syncwarp();
                slab.put(sub, tw[k], tr[k]);
                __syncwarp();
                float part[LPR][4];
                if constexpr (TPG < LPR) {
#pragma unroll
                    for (int j = TPG; j < LPR; ++j) part[j][0] = part[j][1] = part[j][2] = part[j][3] = 0.f;
                }
#pragma unroll
                for (int j = 0; j < TPG; ++j) {
                    const float4 w4 = slab.weights(j);
                    const int2 rr = slab.rows(j);
                    const float w[4] = {w4.x, w4.y, w4.z, w4.w};
                    const unsigned dwo = (rr.y < 0) ? row_elems : 0u;
                    const bool fine = MIXED && rr.x < 0;
                    unsigned long long off[4];
                    off[0] = (unsigned long long)(unsigned)(rr.x & 0x7fffffff) * row_elems;
                    off[1] = off[0] + dwo;
                    off[2] = (unsigned long long)(unsigned)(rr.y & 0x7fffffff) * row_elems;
                    off[3] = off[2] + dwo;
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        float v[VEC];
                        RowVec<T, VEC>::load(base + off[c], v);
                        float dsum = 0.f;
#pragma unroll
                        for (int e = 0; e < VEC; ++e) dsum = fmaf(g[e], v[e], dsum);
                        part[j][c] = dsum;
                        if constexpr (DET) {
                            if (w[c] != 0.f) {
                                const size_t row = slab_off - (size_t)sub * VEC + off[c] + (size_t)sub;
#pragma unroll
                                for (int k = 0; k < VEC; ++k)
                                    det_add(ds, det_acc + kDetHeaderWords, grad_value, row + (size_t)k * LPR,
                                            det_contrib(w[c], gt[k]));
                            }
                        } else if constexpr (MIXED) {        // predicated, branch-free: bf16 result row or fp32 scratch row
                            const bool nz = w[c] != 0.f;
                            red_add_mixed(nz && fine, grad_value_bf16 + slab_off + off[c], nz && !fine, gbase + off[c],
                                          w[c] * g[0], w[c] * g[1], w[c] * g[2], w[c] * g[3]);
                        } else if (w[c] != 0.f) {     // masked-out corners, dead taps and idle groups carry weight 0
#pragma unroll
                            for (int e = 0; e < VEC; e += 4)
                                red_add_v4(gbase + off[c] + e, w[c] * g[e], w[c] * g[e + 1], w[c] * g[e + 2],
                                           w[c] * g[e + 3]);
                        }
                    }
                }
                float dot[4];
                group_reduce_scatter<LPR>(part, sub, dot);

                // ---- the lane that resolved the tap finishes it ----
                const int s = SPLIT ? grp * TPG + sub : sub + k * LPR;
                if ((!SPLIT || sub < TPG) && s < LP && active) {
                    const unsigned mk = tmeta[k];
                    const int l = (int)(mk >> 4);
                    const float d0 = (mk & 1u) ? dot[0] : 0.f, d1 = (mk & 2u) ? dot[1] : 0.f;
                    const float d2 = (mk & 4u) ? dot[2] : 0.f, d3 = (mk & 8u) ? dot[3] : 0.f;
                    const float lh = tlh[k], lw = tlw[k], hh = 1.f - lh, hw = 1.f - lw;
                    const float val = hh * hw * d0 + hh * lw * d1 + lh * hw * d2 + lh * lw * d3;   // cuh:155-156
                    const float gw = hh * (d1 - d0) + lh * (d3 - d2);                               // cuh:124,133,142,151
                    const float gh = hw * (d2 - d0) + lw * (d3 - d1);                               // cuh:123,132,141,150
                    const size_t t = (size_t)pair * LP + s;
                    grad_attn[t] = val;
                    const float a = ta[k];
                    reinterpret_cast<float2 *>(grad_loc)[t] =
                        make_float2((float)wm.W[l] * a * gw, (float)wm.H[l] * a * gh);              // cuh:157-158
                }
            }
        }
    }
}

}  // namespace msda
