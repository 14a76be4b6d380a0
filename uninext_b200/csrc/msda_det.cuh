// msda_det.cuh -- deterministic grad_value accumulation for the backward kernels (msda_backward_det_*).
//
// grad_value rows collect their contributions through atomics whose order changes from run to run, so an fp32 sum
// differs in its last bits between runs.  Here every contribution is quantised to a 64-bit fixed-point integer and
// added with integer reds: integer addition is associative, so the sum -- and the result -- no longer depends on the
// order, the schedule, the kernel family (tiled / generic, SPLIT, TMA) or the GPU.
//
// Quantum.  A = max |attn| and G = max |grad_out| over the finite inputs (msda_det_scale).  With A < 2^ea and
// G < 2^eg (frexp exponents), a contribution x = fl(fl(cw * a) * g) with corner weight cw in [0, 1] obeys
// |x| <= fl(A * G) <= 2^e, e = ea + eg (rounding is monotone and 2^e is representable).  A value row receives at most
// K = Lq * L * P contributions.  With c = ceil(log2 K) and the scale 2^s, s = 62 - c - e, every quantised term is at most
// 2^(62 - c) in magnitude and every partial sum, in any order, at most 2^62: no int64 overflow.  The quantum 2^-s is
// 2^(e + c - 62), i.e. about 2^-43 * A * G at the cfg2 encoder call (K ~ 2^19), far below fp32 rounding of the sums.
// The scaling runs in fp64, where x * 2^s is exact for every fp32 x and every s this bound produces.
//
// Non-finite inputs.  A NaN / Inf contribution cannot be quantised.  When the scale pass saw a non-finite attn or
// grad_out (or A * G may overflow fp32), the kernels take a uniform branch that adds the non-finite contributions with
// fp32 atomics into the (then zero-filled) output buffer; an IEEE sum of only non-finite terms does not depend on its
// order.  The convert pass adds that buffer to the fixed-point result.
//
// Accumulator layout: kDetHeaderWords int64 header words (A bits, G bits, non-finite flag, pad), then N*S*M*D sums.
#pragma once

#include "msda_common.cuh"

namespace msda {

constexpr int kDetHeaderWords = 4;     // keeps the sums 32-byte aligned when the buffer is

// The one canonical fp32 contribution of a tap corner to a grad_value element: masked corner weight (cw * a, see
// masked_weights) times the output gradient.  Every kernel family calls this in deterministic mode.
__device__ __forceinline__ float det_contrib(float w, float g) { return __fmul_rn(w, g); }

struct DetScale {
    double scale;        // 2^s
    double quantum;      // 2^-s
    bool nonfinite;      // take the non-finite branch
};

__device__ __forceinline__ int frexp_exp(float v) { return v > 0.f ? ilogbf(v) + 1 : 0; }

__device__ __forceinline__ DetScale det_scale(const unsigned long long *hdr, int clog2) {
    const float A = __uint_as_float((unsigned)hdr[0]), G = __uint_as_float((unsigned)hdr[1]);
    const int e = (A > 0.f && G > 0.f) ? frexp_exp(A) + frexp_exp(G) : 0;
    DetScale d;
    d.scale = ldexp(1.0, 62 - clog2 - e);
    d.quantum = ldexp(1.0, e + clog2 - 62);
    d.nonfinite = hdr[2] != 0ull || e >= 128;          // e >= 128: a finite product may round to Inf
    return d;
}

__device__ __forceinline__ void red_add_u64(unsigned long long *addr, long long v) {
    asm volatile("red.global.add.u64 [%0], %1;" ::"l"(addr), "l"(v) : "memory");
}

// Adds contribution x to element `i` of the fixed-point sums (or, in the non-finite branch, a non-finite x to nf[i]).
__device__ __forceinline__ void det_add(const DetScale &ds, unsigned long long *sums, float *nf, size_t i, float x) {
    if (ds.nonfinite && !isfinite(x)) {
        atomicAdd(nf + i, x);
        return;
    }
    red_add_u64(sums + i, __double2ll_rn((double)x * ds.scale));
}

// Scale pass: max |attn| and max |grad_out| over the finite entries (integer max on the bits of non-negative floats is
// exact), plus the non-finite flag.  hdr must be zero on entry.
template <typename T>
__global__ void __launch_bounds__(256)
msda_det_scale(const float *__restrict__ attn, long long n_attn, const T *__restrict__ grad_out, long long n_go,
               unsigned long long *__restrict__ hdr) {
    unsigned am = 0u, gm = 0u, bad = 0u;
    const long long stride = (long long)gridDim.x * blockDim.x;
#pragma unroll 1
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_attn; i += stride) {
        const float v = fabsf(attn[i]);
        if (isfinite(v)) am = max(am, __float_as_uint(v)); else bad = 1u;
    }
#pragma unroll 1
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_go; i += stride) {
        const float v = fabsf((float)grad_out[i]);
        if (isfinite(v)) gm = max(gm, __float_as_uint(v)); else bad = 1u;
    }
    __shared__ unsigned s_am[8], s_gm[8], s_bad[8];                      // one set of atomics per CTA, not per warp
    am = __reduce_max_sync(kFullMask, am);
    gm = __reduce_max_sync(kFullMask, gm);
    bad = __reduce_or_sync(kFullMask, bad);
    if ((threadIdx.x & 31) == 0) { s_am[threadIdx.x >> 5] = am; s_gm[threadIdx.x >> 5] = gm; s_bad[threadIdx.x >> 5] = bad; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) { am = max(am, s_am[w]); gm = max(gm, s_gm[w]); bad |= s_bad[w]; }
        if (am) atomicMax(hdr + 0, (unsigned long long)am);
        if (gm) atomicMax(hdr + 1, (unsigned long long)gm);
        if (bad) atomicOr(hdr + 2, 1ull);
    }
}

// Zero-fills the non-finite buffer, only when the scale pass took the non-finite branch (otherwise the convert pass
// overwrites every element and the buffer needs no fill).
__global__ void __launch_bounds__(256)
msda_det_prepare(const unsigned long long *__restrict__ hdr, int clog2, float *__restrict__ nf, long long n) {
    if (!det_scale(hdr, clog2).nonfinite) return;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        nf[i] = 0.f;
}

// Convert pass: out = fp32(sum * quantum) (+ the non-finite buffer), and / or its bf16 rounding.
__global__ void __launch_bounds__(256)
msda_det_convert(const unsigned long long *__restrict__ hdr, int clog2, const float *nf, long long n, float *out32,
                 __nv_bfloat16 *__restrict__ out16) {
    const DetScale ds = det_scale(hdr, clog2);
    const long long *sums = reinterpret_cast<const long long *>(hdr + kDetHeaderWords);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        float v = (float)((double)sums[i] * ds.quantum);
        if (ds.nonfinite) v += nf[i];
        if (out32) out32[i] = v;
        if (out16) out16[i] = __float2bfloat16_rn(v);
    }
}

}  // namespace msda
