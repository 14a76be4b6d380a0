// msda_generic.cuh -- shape-agnostic kernels (any D, L, P; fp64 / fp32 / bf16 storage).
//
// They exist so the library is a complete drop-in: the reference op accepts any channel count and double precision
// (its own test gradchecks D in {30,32,64,71,1025,2048,3096} in fp64, ops/test.py:63-86).  Production shapes
// (D multiple of the 16-byte vector, L <= 8, L*P <= 32) never reach this file -- see msda_cabi.cu:route().
#pragma once

#include "msda_common.cuh"
#include "msda_det.cuh"

namespace msda {

// storage <-> compute conversions (compute type C is double for fp64 storage, float otherwise)
template <typename T> struct Num;
template <> struct Num<double> { using C = double; __device__ static double ld(const double *p) { return __ldg(p); } __device__ static void st(double *p, double v) { *p = v; } };
template <> struct Num<float> { using C = float; __device__ static float ld(const float *p) { return __ldg(p); } __device__ static void st(float *p, float v) { *p = v; } };
template <> struct Num<__nv_bfloat16> {
    using C = float;
    __device__ static float ld(const __nv_bfloat16 *p) { return __bfloat162float(*p); }
    __device__ static void st(__nv_bfloat16 *p, float v) { *p = __float2bfloat16_rn(v); }
};

template <typename C>
struct GTap {
    C lh, lw;
    long long r[4];     // row index per corner, -1 when the corner is outside the map
    bool inside;
};

template <typename C>
__device__ __forceinline__ GTap<C> generic_tap(C x, C y, int H, int W, long long start) {
    GTap<C> t;
    const C h_im = y * (C)H - (C)0.5;                       // cuh:285
    const C w_im = x * (C)W - (C)0.5;                       // cuh:286
    t.inside = (h_im > (C)-1) && (w_im > (C)-1) && (h_im < (C)H) && (w_im < (C)W);      // cuh:288
    const C hf = floor(h_im), wf = floor(w_im);
    t.lh = h_im - hf; t.lw = w_im - wf;
    const int h0 = t.inside ? (int)hf : 0, w0 = t.inside ? (int)wf : 0, h1 = h0 + 1, w1 = w0 + 1;
    const bool top = h0 >= 0, bot = h1 <= H - 1, lef = w0 >= 0, rig = w1 <= W - 1;
    t.r[0] = (t.inside && top && lef) ? start + (long long)h0 * W + w0 : -1;
    t.r[1] = (t.inside && top && rig) ? start + (long long)h0 * W + w1 : -1;
    t.r[2] = (t.inside && bot && lef) ? start + (long long)h1 * W + w0 : -1;
    t.r[3] = (t.inside && bot && rig) ? start + (long long)h1 * W + w1 : -1;
    return t;
}

// One thread per output element (pair, channel); channel fastest so a warp reads contiguous row slices.
template <typename T, typename TL>
__global__ void __launch_bounds__(256)
msda_fwd_generic(const T *__restrict__ value, const int64_t *__restrict__ shapes, const int64_t *__restrict__ lsi,
                 const TL *__restrict__ loc, const TL *__restrict__ attn,
                 int S, int M, int D, int L, int Lq, int P, long long total, T *__restrict__ out)
{
    using C = typename Num<T>::C;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(idx % D);
        const long long pair = idx / D;
        const int m = (int)(pair % M);
        const long long b = (pair / M) / Lq;
        const size_t row_elems = (size_t)M * D;
        const T *slab = value + (size_t)b * S * row_elems + (size_t)m * D + c;
        C acc = 0;
        for (int l = 0; l < L; ++l) {
            const int H = (int)shapes[2 * l], W = (int)shapes[2 * l + 1];
            const long long start = lsi[l];
            for (int p = 0; p < P; ++p) {
                const long long t = (pair * L + l) * P + p;
                const GTap<C> g = generic_tap<C>((C)loc[2 * t], (C)loc[2 * t + 1], H, W, start);
                if (!g.inside) continue;
                const C hh = (C)1 - g.lh, hw = (C)1 - g.lw;
                const C v0 = g.r[0] >= 0 ? Num<T>::ld(slab + (size_t)g.r[0] * row_elems) : (C)0;
                const C v1 = g.r[1] >= 0 ? Num<T>::ld(slab + (size_t)g.r[1] * row_elems) : (C)0;
                const C v2 = g.r[2] >= 0 ? Num<T>::ld(slab + (size_t)g.r[2] * row_elems) : (C)0;
                const C v3 = g.r[3] >= 0 ? Num<T>::ld(slab + (size_t)g.r[3] * row_elems) : (C)0;
                acc += (hh * hw * v0 + hh * g.lw * v1 + g.lh * hw * v2 + g.lh * g.lw * v3) * (C)attn[t];
            }
        }
        Num<T>::st(out + idx, acc);
    }
}

template <typename C>
__device__ __forceinline__ C block_sum(C v, C *scratch) {
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) v += __shfl_xor_sync(kFullMask, v, d);
    const int warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    __syncthreads();                      // scratch reuse across calls
    if ((threadIdx.x & 31) == 0) scratch[warp] = v;
    __syncthreads();
    C tot = 0;
    for (int i = 0; i < nw; ++i) tot += scratch[i];
    return tot;
}

// One block per (b,q,m) pair, threads stride over channels.  GA is the grad_value accumulator type
// (T for fp32/fp64, float for bf16 storage).
// DET (fp32 compute only, msda_det.cuh): grad_value goes to the fixed-point sums in det_acc, from the tiled kernels' tap
// geometry, skip rule and fp32 products, so both families produce the same bits; grad_value only receives non-finite
// contributions.
template <typename T, typename TL, typename GA, bool DET = false>
__global__ void __launch_bounds__(256)
msda_bwd_generic(const T *__restrict__ grad_out, const T *__restrict__ value,
                 const int64_t *__restrict__ shapes, const int64_t *__restrict__ lsi,
                 const TL *__restrict__ loc, const TL *__restrict__ attn,
                 int S, int M, int D, int L, int Lq, int P, long long npairs,
                 GA *__restrict__ grad_value, TL *__restrict__ grad_loc, TL *__restrict__ grad_attn,
                 unsigned long long *__restrict__ det_acc, int det_clog2)
{
    using C = typename Num<T>::C;
    static_assert(!DET || sizeof(C) == 4, "DET: fp32 contributions");
    __shared__ C scratch[8];
    DetScale ds{};
    if constexpr (DET) ds = det_scale(det_acc, det_clog2);
    for (long long pair = blockIdx.x; pair < npairs; pair += gridDim.x) {
        const int m = (int)(pair % M);
        const long long b = (pair / M) / Lq;
        const size_t row_elems = (size_t)M * D;
        const size_t slab = (size_t)b * S * row_elems + (size_t)m * D;
        for (int l = 0; l < L; ++l) {
            const int H = (int)shapes[2 * l], W = (int)shapes[2 * l + 1];
            const long long start = lsi[l];
            for (int p = 0; p < P; ++p) {
                const long long t = (pair * L + l) * P + p;
                const C a = (C)attn[t];
                const GTap<C> g = generic_tap<C>((C)loc[2 * t], (C)loc[2 * t + 1], H, W, start);
                if constexpr (DET) {
                    const TapGeom gm = tap_geometry((float)loc[2 * t], (float)loc[2 * t + 1], H, W, (int)start);
                    const float4 w4 = masked_weights(gm, (float)a);
                    const float w[4] = {w4.x, w4.y, w4.z, w4.w};
                    const size_t row[4] = {slab + (size_t)gm.r0 * row_elems, slab + (size_t)(gm.r0 + gm.dw) * row_elems,
                                           slab + (size_t)gm.r1 * row_elems, slab + (size_t)(gm.r1 + gm.dw) * row_elems};
                    if (gm.mask) {
                        for (int c = threadIdx.x; c < D; c += blockDim.x) {
                            const float go = Num<T>::ld(grad_out + (size_t)pair * D + c);
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                if (w[k] != 0.f)
                                    det_add(ds, det_acc + kDetHeaderWords, grad_value, row[k] + c, det_contrib(w[k], go));
                        }
                    }
                }
                C ga = 0, gx = 0, gy = 0;
                if (g.inside) {
                    const C hh = (C)1 - g.lh, hw = (C)1 - g.lw;
                    const C cw[4] = {hh * hw, hh * g.lw, g.lh * hw, g.lh * g.lw};
                    for (int c = threadIdx.x; c < D; c += blockDim.x) {
                        const C go = Num<T>::ld(grad_out + (size_t)pair * D + c);
                        C v[4];
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            v[k] = 0;
                            if (g.r[k] >= 0) {
                                const size_t o = slab + (size_t)g.r[k] * row_elems + c;
                                v[k] = Num<T>::ld(value + o);
                                if constexpr (!DET) atomicAdd(grad_value + o, (GA)(cw[k] * a * go));   // cuh:125,134,143,152
                            }
                        }
                        ga += go * (cw[0] * v[0] + cw[1] * v[1] + cw[2] * v[2] + cw[3] * v[3]);     // cuh:156
                        gx += go * (hh * (v[1] - v[0]) + g.lh * (v[3] - v[2]));                      // cuh:157
                        gy += go * (hw * (v[2] - v[0]) + g.lw * (v[3] - v[1]));                      // cuh:158
                    }
                }
                ga = block_sum<C>(ga, scratch);
                gx = block_sum<C>(gx, scratch);
                gy = block_sum<C>(gy, scratch);
                if (threadIdx.x == 0) {
                    grad_attn[t] = (TL)ga;
                    grad_loc[2 * t] = (TL)((C)W * a * gx);
                    grad_loc[2 * t + 1] = (TL)((C)H * a * gy);
                }
            }
        }
    }
}

// fp32 accumulator -> bf16 result (bf16 backward only)
__global__ void __launch_bounds__(256)
msda_f32_to_bf16(const float *__restrict__ src, __nv_bfloat16 *__restrict__ dst, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        dst[i] = __float2bfloat16_rn(src[i]);
}

// Mixed bf16 backward (msda_bwd_tiled, MIXED): rows of the COARSE levels (H_l * W_l < fine_min_rows) are accumulated in
// the fp32 scratch and rounded into the bf16 result afterwards; rows of the fine levels never touch the scratch.  Both
// helpers walk the rows of one batch element per blockIdx.y and read the level table on the device.
//   ROUND = false: zero the scratch rows of the coarse levels (before the backward kernel);
//   ROUND = true : dst[row] = bf16(scratch[row]) for the coarse levels (after it).
template <bool ROUND>
__global__ void __launch_bounds__(256)
msda_coarse_rows(float *__restrict__ scratch, __nv_bfloat16 *__restrict__ dst, const int64_t *__restrict__ shapes,
                 const int64_t *__restrict__ lsi, int L, int S, int row_elems, int fine_min_rows) {
    const int b = blockIdx.y;
    const int quads = row_elems / 4;
    for (int l = 0; l < L; ++l) {
        const int rows = (int)(shapes[2 * l] * shapes[2 * l + 1]);
        if (rows >= fine_min_rows) continue;
        const long long first = ((long long)b * S + (int)lsi[l]) * row_elems;
        const long long n4 = (long long)rows * quads;
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
            float4 *p = reinterpret_cast<float4 *>(scratch + first) + i;
            if (ROUND) {
                const float4 v = *p;
                const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
                reinterpret_cast<uint2 *>(dst + first)[i] = make_uint2(*reinterpret_cast<const unsigned *>(&lo),
                                                                      *reinterpret_cast<const unsigned *>(&hi));
            } else {
                *p = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
    }
}

}  // namespace msda
