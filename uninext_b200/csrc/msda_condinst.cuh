// msda_condinst.cuh -- CondInst dynamic mask head (SURVEY.md section 8 f-4), the mask branch of UNINEXT's video / instance
// configs (uninext/models/ddetrs.py:488-598 `mask_heads_forward` + `dynamic_mask_with_coords`, :895-944 helpers).
//
// Reference formulation: for every selected instance a 3-layer MLP of 1x1 convolutions whose 169 weights come from the
// controller (10 -> 8 -> 8 -> 1 channels; input = 2 relative coordinates + the 8 mask-feature channels of the instance's
// image), evaluated at every pixel of the stride-8 mask feature map.  The reference materialises the input as
// [1, I * 10, H, W] with `repeat` (201 MB for 300 instances at 100 x 168) and runs three grouped convolutions with
// groups = I -- a shape cuDNN handles badly -- then upsamples with `aligned_bilinear`.
//
// Here: a thread keeps 4 (forward) / 2 (backward) consecutive pixels -- their 8 feature channels and locations -- in
// registers as packed fp32 pairs and loops over a chunk of 16 instances of its image, whose parameters sit in shared
// memory (broadcast reads); the work is the fp32 pipe's (152 FMA per pixel and instance forward).  Nothing is materialised.
//   forward : logits[i, y, x]                                         (ddetrs.py:493-505, 523-566)
//   backward: recomputes the hidden activations; grad_feats summed over the chunk in registers, one RED per value and
//             chunk; the 171 per-instance sums over pixels (169 parameters + 2 reference coordinates) use a transposing
//             warp reduction (16 shuffles per 16 values instead of 80) and one RED per group -- no block barrier inside
//             the instance loop.
//   aligned_bilinear forward / backward (ddetrs.py:921-942): replicate-pad, align_corners bilinear x factor, shift by
//   factor / 2 -- closed form, gather on both passes, four outputs per thread on the forward pass.
// Parameter layout of one instance (parse_dynamic_params, ddetrs.py:895-918): w1[8][10] | w2[8][8] | w3[8] | b1[8] | b2[8] | b3,
// input channel order (rel_x, rel_y, feat_0..7) with rel = reference_point - (pixel * stride + stride / 2)  (:533-541, :944-958).
#pragma once

#include "msda_common.cuh"

namespace msda {

constexpr int kCiFeat = 8;                  // mask feature channels (hidden_dim / 32)
constexpr int kCiCh = 8;                    // dynamic_mask_channels
constexpr int kCiIn = kCiFeat + 2;
constexpr int kCiParams = kCiCh * kCiIn + kCiCh * kCiCh + kCiCh + kCiCh + kCiCh + 1;      // 169
constexpr int kCiW1 = 0, kCiW2 = kCiCh * kCiIn, kCiW3 = kCiW2 + kCiCh * kCiCh, kCiB1 = kCiW3 + kCiCh, kCiB2 = kCiB1 + kCiCh,
              kCiB3 = kCiB2 + kCiCh;
constexpr int kCiSums = kCiParams + 2;      // per-instance sums of the backward pass: parameters, then d/d(ref_x, ref_y)
constexpr int kCiRow = kCiParams + 3;       // shared-memory row: parameters, ref_x, ref_y, pad
constexpr int kCiThreads = 128;             // backward
constexpr int kCiFwdThreads = 128;          // forward
constexpr int kCiChunk = 16;                // instances whose parameters are staged in shared memory at a time
constexpr int kCiFwdGroups = 1;             // forward: groups of 4 pixels per thread (2: same time at 190 registers)
constexpr int kCiFwdPpt = 4 * kCiFwdGroups, kCiBwdPpt = 2;      // pixels per thread

// ---- packed fp32 pairs (FFMA2 = `fma.rn.f32x2`): the kernels keep two neighbouring pixels in the halves of a 64-bit register
// pair.  A pair built from the same scalar twice compiles to FFMA2's scalar-broadcast operand, so a parameter costs one
// 32-bit register read for two FMAs.  Measured issue cost per scheduler (tools/ubench_ffma.cu): FFMA with three registers
// 1.5 cycles, FFMA2 with a broadcast multiplier 2.25 cycles per TWO FMAs -- the register file's read ports, not the fp32
// lanes, set the rate -- and half the issue slots are left for the shared-memory reads of the parameters.
struct f2 { unsigned long long v; };
__device__ __forceinline__ f2 f2_make(float lo, float hi) { f2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r.v) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ f2 f2_bcast(float a) { return f2_make(a, a); }
__device__ __forceinline__ float f2_lo(f2 a) { float lo, hi; asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a.v)); return lo; }
__device__ __forceinline__ float f2_hi(f2 a) { float lo, hi; asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a.v)); return hi; }
__device__ __forceinline__ f2 f2_fma(f2 a, f2 b, f2 c) { f2 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r.v) : "l"(a.v), "l"(b.v), "l"(c.v)); return r; }
__device__ __forceinline__ f2 f2_mul(f2 a, f2 b) { f2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v)); return r; }
__device__ __forceinline__ f2 f2_relu(f2 a) { return f2_make(fmaxf(f2_lo(a), 0.f), fmaxf(f2_hi(a), 0.f)); }
// a where the matching half of m is positive, else 0
__device__ __forceinline__ f2 f2_gate(f2 a, f2 m) { return f2_make(f2_lo(m) > 0.f ? f2_lo(a) : 0.f, f2_hi(m) > 0.f ? f2_hi(a) : 0.f); }

// The three layers on pairs.  wf(j) returns parameter j as a pair (broadcast of one instance's value, or two instances'
// values), xf(q, c) layer-1 input c of pair q; h1 / h2 = post-ReLU activations.
template <int NP, class WF, class XF>
__device__ __forceinline__ void ci_forward(WF wf, XF xf, f2 (&h1)[NP][kCiCh], f2 (&h2)[NP][kCiCh], f2 (&out)[NP]) {
#pragma unroll
    for (int o = 0; o < kCiCh; ++o) {
        f2 a[NP];
        const f2 bias = wf(kCiB1 + o);
#pragma unroll
        for (int q = 0; q < NP; ++q) a[q] = bias;
#pragma unroll
        for (int c = 0; c < kCiIn; ++c) {
            const f2 wt = wf(kCiW1 + o * kCiIn + c);
#pragma unroll
            for (int q = 0; q < NP; ++q) a[q] = f2_fma(wt, xf(q, c), a[q]);
        }
#pragma unroll
        for (int q = 0; q < NP; ++q) h1[q][o] = f2_relu(a[q]);
    }
#pragma unroll
    for (int o = 0; o < kCiCh; ++o) {
        f2 a[NP];
        const f2 bias = wf(kCiB2 + o);
#pragma unroll
        for (int q = 0; q < NP; ++q) a[q] = bias;
#pragma unroll
        for (int c = 0; c < kCiCh; ++c) {
            const f2 wt = wf(kCiW2 + o * kCiCh + c);
#pragma unroll
            for (int q = 0; q < NP; ++q) a[q] = f2_fma(wt, h1[q][c], a[q]);
        }
#pragma unroll
        for (int q = 0; q < NP; ++q) h2[q][o] = f2_relu(a[q]);
    }
    const f2 b3 = wf(kCiB3);
#pragma unroll
    for (int q = 0; q < NP; ++q) out[q] = b3;
#pragma unroll
    for (int c = 0; c < kCiCh; ++c) {
        const f2 wt = wf(kCiW3 + c);
#pragma unroll
        for (int q = 0; q < NP; ++q) out[q] = f2_fma(wt, h2[q][c], out[q]);
    }
}

// Forward-only variant: layer 3 folded into layer 2's output loop, so h2 is never held (same summation order).
template <int NP, class WF, class XF>
__device__ __forceinline__ void ci_forward_logit(WF wf, XF xf, f2 (&out)[NP]) {
    f2 h1[NP][kCiCh];
#pragma unroll
    for (int o = 0; o < kCiCh; ++o) {
        f2 a[NP];
        const f2 bias = wf(kCiB1 + o);
#pragma unroll
        for (int q = 0; q < NP; ++q) a[q] = bias;
#pragma unroll
        for (int c = 0; c < kCiIn; ++c) {
            const f2 wt = wf(kCiW1 + o * kCiIn + c);
#pragma unroll
            for (int q = 0; q < NP; ++q) a[q] = f2_fma(wt, xf(q, c), a[q]);
        }
#pragma unroll
        for (int q = 0; q < NP; ++q) h1[q][o] = f2_relu(a[q]);
    }
    const f2 b3 = wf(kCiB3);
#pragma unroll
    for (int q = 0; q < NP; ++q) out[q] = b3;
#pragma unroll
    for (int o = 0; o < kCiCh; ++o) {
        f2 a[NP];
        const f2 bias = wf(kCiB2 + o);
#pragma unroll
        for (int q = 0; q < NP; ++q) a[q] = bias;
#pragma unroll
        for (int c = 0; c < kCiCh; ++c) {
            const f2 wt = wf(kCiW2 + o * kCiCh + c);
#pragma unroll
            for (int q = 0; q < NP; ++q) a[q] = f2_fma(wt, h1[q][c], a[q]);
        }
        const f2 w3 = wf(kCiW3 + o);
#pragma unroll
        for (int q = 0; q < NP; ++q) out[q] = f2_fma(w3, f2_relu(a[q]), out[q]);
    }
}

__device__ __forceinline__ float ci_loc(int px, int W, int stride, bool want_y) {
    return (float)((want_y ? px / W : px % W) * stride + stride / 2);
}

// ---- forward: a pair = two neighbouring pixels of one instance; a thread owns kCiFwdGroups groups of 4 consecutive pixels,
// group g of thread t at pixel (tile * groups + g) * 4 * blockDim + 4 * t, so every 16-byte access of a warp is contiguous.
// grid: (pixel tiles, instance chunks, images).  feats [N, 8, H*W]; params [I, 169]; refs [I, 2] (pixels of the input image);
// inst_start [N + 1] (instances of image b are [inst_start[b], inst_start[b + 1])); logits [I, H*W].
__global__ void __launch_bounds__(kCiFwdThreads)
condinst_fwd(const float *__restrict__ feats, const float *__restrict__ params, const float *__restrict__ refs,
             const int *__restrict__ inst_start, int HW, int W, int stride, int rel_coord, float *__restrict__ logits)
{
    constexpr int G = kCiFwdGroups, NP = 2 * G;
    __shared__ __align__(16) float sp[kCiChunk][kCiRow];
    const int b = blockIdx.z;
    const int i0 = inst_start[b] + blockIdx.y * kCiChunk, i1 = min(inst_start[b + 1], i0 + kCiChunk);
    if (i0 >= i1) return;
    for (int t = threadIdx.x; t < (i1 - i0) * kCiSums; t += kCiFwdThreads) {
        const int k = t / kCiSums, j = t - k * kCiSums;
        sp[k][j] = j < kCiParams ? params[(size_t)(i0 + k) * kCiParams + j] : refs[(size_t)(i0 + k) * 2 + (j - kCiParams)];
    }
    __syncthreads();
    int gpx[G];                                 // first pixel of each group
#pragma unroll
    for (int g = 0; g < G; ++g) gpx[g] = ((blockIdx.x * G + g) * kCiFwdThreads + threadIdx.x) * 4;
    if (gpx[0] >= HW) return;
    const bool vec = (HW & 3) == 0;            // then a live group has 4 pixels and every row of feats / logits is 16-byte aligned
    f2 x[NP][kCiIn], lx[NP], ly[NP];
#pragma unroll
    for (int g = 0; g < G; ++g) {
#pragma unroll
        for (int c = 0; c < kCiFeat; ++c) {
            const float *src = feats + ((size_t)b * kCiFeat + c) * HW + gpx[g];
            float v[4];
            if (vec && gpx[g] < HW) {
                const float4 t = __ldg(reinterpret_cast<const float4 *>(src));
                v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q) v[q] = gpx[g] + q < HW ? __ldg(src + q) : 0.f;
            }
            x[2 * g][2 + c] = f2_make(v[0], v[1]);
            x[2 * g + 1][2 + c] = f2_make(v[2], v[3]);
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int pa = min(gpx[g] + 2 * q, HW - 1), pb = min(gpx[g] + 2 * q + 1, HW - 1);
            lx[2 * g + q] = f2_make(ci_loc(pa, W, stride, false), ci_loc(pb, W, stride, false));
            ly[2 * g + q] = f2_make(ci_loc(pa, W, stride, true), ci_loc(pb, W, stride, true));
        }
    }
    const f2 minus1 = f2_bcast(-1.f), zero = f2_bcast(0.f);
    for (int k = 0; k < i1 - i0; ++k) {
        const float *p = sp[k];
        auto wf = [p](int j) { return f2_bcast(p[j]); };
#pragma unroll
        for (int q = 0; q < NP; ++q) {
            x[q][0] = rel_coord ? f2_fma(minus1, lx[q], wf(kCiParams)) : zero;          // ref - location, one rounding
            x[q][1] = rel_coord ? f2_fma(minus1, ly[q], wf(kCiParams + 1)) : zero;
        }
        f2 out[NP];
        ci_forward_logit<NP>(wf, [&x](int q, int c) { return x[q][c]; }, out);
#pragma unroll
        for (int g = 0; g < G; ++g) {
            float *dst = logits + (size_t)(i0 + k) * HW + gpx[g];
            if (vec) {
                if (gpx[g] < HW)
                    *reinterpret_cast<float4 *>(dst) = make_float4(f2_lo(out[2 * g]), f2_hi(out[2 * g]), f2_lo(out[2 * g + 1]), f2_hi(out[2 * g + 1]));
            } else {
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    if (gpx[g] + 2 * q < HW) dst[2 * q] = f2_lo(out[2 * g + q]);
                    if (gpx[g] + 2 * q + 1 < HW) dst[2 * q + 1] = f2_hi(out[2 * g + q]);
                }
            }
        }
    }
}

// Transposing warp reduction over NV values per lane (NV = 16 here): step d halves the live set -- a lane keeps the half
// whose index bit matches its own lane bit and receives the partner's copy of that half (8 + 4 + 2 + 1 shuffles); the
// last shuffle folds lanes l and l ^ 16.  On return every lane holds the warp-wide sum of v[lane % 16].
__device__ __forceinline__ float warp_transpose_sum16(float (&v)[16], int lane) {
#pragma unroll
    for (int d = 8; d >= 1; d >>= 1) {
        const bool hi = (lane & d) != 0;
#pragma unroll
        for (int i = 0; i < d; ++i) {
            const float send = hi ? v[i] : v[i + d];
            const float keep = hi ? v[i + d] : v[i];
            v[i] = keep + __shfl_xor_sync(kFullMask, send, d);
        }
    }
    return v[0] + __shfl_xor_sync(kFullMask, v[0], 16);
}

// ---- backward: same pairing as the forward pass (two neighbouring pixels of one instance), one pair per thread.
// Recomputes the activations, then
//   d2 / d1 = gradients wrt the pre-activations of layers 2 / 1, dx = gradient wrt the layer-1 input (features: summed over
//   the chunk in registers, one RED per value at the end);
//   the 171 per-instance sums over pixels (169 parameters + d/d(ref_x, ref_y)) in 11 groups of 16, each group as soon as
//   its operands exist so that h2, then h1, die early: product per pixel pair (FMUL2), the two halves added, transposing
//   warp reduction, one RED per group from lanes 0-15.
// grid: (pixel tiles, instance chunks, images).  grad_feats [N, 8, H*W], grad_params [I, 169] and grad_refs [I, 2] must be
// zero on entry.
// DET: no atomics.  Each thread stores its chunk's feature gradient to feat_part [chunk][N][8][H*W], and each warp stores its
// 171 per-instance sums to sum_part [warp slot][I][171] (warp slot = global warp index, 64 pixels each); condinst_bwd_reduce
// then adds the partials in a fixed order.
template <bool DET = false>
__global__ void __launch_bounds__(kCiThreads, 3)
condinst_bwd(const float *__restrict__ grad_logits, const float *__restrict__ feats, const float *__restrict__ params,
             const float *__restrict__ refs, const int *__restrict__ inst_start, int HW, int W, int stride, int rel_coord,
             float *__restrict__ grad_feats, float *__restrict__ grad_params, float *__restrict__ grad_refs,
             float *__restrict__ feat_part = nullptr, float *__restrict__ sum_part = nullptr, int I = 0)
{
    static_assert(kCiBwdPpt == 2, "one pixel pair per thread");
    __shared__ __align__(16) float sp[kCiChunk][kCiRow];
    const int b = blockIdx.z;
    const int i0 = inst_start[b] + blockIdx.y * kCiChunk, i1 = min(inst_start[b + 1], i0 + kCiChunk);
    if (i0 >= i1) return;
    for (int t = threadIdx.x; t < (i1 - i0) * kCiSums; t += kCiThreads) {
        const int k = t / kCiSums, j = t - k * kCiSums;
        sp[k][j] = j < kCiParams ? params[(size_t)(i0 + k) * kCiParams + j] : refs[(size_t)(i0 + k) * 2 + (j - kCiParams)];
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int px0 = (blockIdx.x * kCiThreads + threadIdx.x) * 2;
    if ((blockIdx.x * kCiThreads + (threadIdx.x & ~31)) * 2 >= HW) return;        // whole warp past the end
    const bool live0 = px0 < HW, live1 = px0 + 1 < HW;
    const int pa = live0 ? px0 : HW - 1, pb = live1 ? px0 + 1 : HW - 1;
    f2 x[1][kCiIn], gf[kCiFeat];
    const f2 lx = f2_make(ci_loc(pa, W, stride, false), ci_loc(pb, W, stride, false));
    const f2 ly = f2_make(ci_loc(pa, W, stride, true), ci_loc(pb, W, stride, true));
    const f2 zero = f2_bcast(0.f), minus1 = f2_bcast(-1.f);
#pragma unroll
    for (int c = 0; c < kCiFeat; ++c) {
        const float *src = feats + ((size_t)b * kCiFeat + c) * HW;
        x[0][2 + c] = f2_make(live0 ? __ldg(src + pa) : 0.f, live1 ? __ldg(src + pb) : 0.f);
        gf[c] = zero;
    }
    auto xf = [&x](int, int c) { return x[0][c]; };

    for (int k = 0; k < i1 - i0; ++k) {
        const float *p = sp[k];
        auto wf = [p](int j) { return f2_bcast(p[j]); };
        x[0][0] = rel_coord ? f2_fma(minus1, lx, wf(kCiParams)) : zero;            // ref - location, one rounding
        x[0][1] = rel_coord ? f2_fma(minus1, ly, wf(kCiParams + 1)) : zero;
        // sums[i] = this thread's pixel pair's terms of 16 sums; lane l < 16 adds the warp total of sums[l] to dst(l) (< 0: none)
        auto reduce_group = [&](const f2 (&sums)[16], auto dst) {
            float v[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = f2_lo(sums[i]) + f2_hi(sums[i]);
            const float sum = warp_transpose_sum16(v, lane);
            const int j = dst(lane & 15);
            if constexpr (DET) {
                const size_t slot = (size_t)(blockIdx.x * (kCiThreads / 32) + (threadIdx.x >> 5));
                if (lane < 16 && j >= 0) sum_part[(slot * I + (i0 + k)) * kCiSums + j] = sum;
            } else if (lane < 16 && j >= 0) {
                if (j < kCiParams) atomicAdd(grad_params + (size_t)(i0 + k) * kCiParams + j, sum);
                else atomicAdd(grad_refs + (size_t)(i0 + k) * 2 + (j - kCiParams), sum);
            }
        };

        f2 h1[1][kCiCh], d2[kCiCh], go;
        {
            f2 h2[1][kCiCh], out[1];
            ci_forward<1>(wf, xf, h1, h2, out);
            const float *gl = grad_logits + (size_t)(i0 + k) * HW;
            go = f2_make(live0 ? __ldg(gl + pa) : 0.f, live1 ? __ldg(gl + pb) : 0.f);
            f2 sums[16];                                                    // w3: go * h2;  b2: d2
#pragma unroll
            for (int c = 0; c < kCiCh; ++c) {
                d2[c] = f2_gate(f2_mul(go, wf(kCiW3 + c)), h2[0][c]);
                sums[c] = f2_mul(go, h2[0][c]);
                sums[8 + c] = d2[c];
            }
            reduce_group(sums, [](int i) { return i < 8 ? kCiW3 + i : kCiB2 + (i - 8); });
        }
        f2 d1[kCiCh];
#pragma unroll
        for (int c = 0; c < kCiCh; ++c) {
            f2 a = zero;
#pragma unroll
            for (int o = 0; o < kCiCh; ++o) a = f2_fma(wf(kCiW2 + o * kCiCh + c), d2[o], a);
            d1[c] = f2_gate(a, h1[0][c]);
        }
#pragma unroll
        for (int g = 0; g < kCiCh * kCiCh / 16; ++g) {                      // w2[o][c]: d2[o] * h1[c]
            f2 sums[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) sums[i] = f2_mul(d2[(g * 16 + i) / kCiCh], h1[0][(g * 16 + i) % kCiCh]);
            reduce_group(sums, [g](int i) { return kCiW2 + g * 16 + i; });
        }
        f2 dx01[2];
#pragma unroll
        for (int c = 0; c < kCiIn; ++c) {
            f2 a = c < 2 ? zero : gf[c < 2 ? 0 : c - 2];
#pragma unroll
            for (int o = 0; o < kCiCh; ++o) a = f2_fma(wf(kCiW1 + o * kCiIn + c), d1[o], a);
            if (c < 2) dx01[c] = rel_coord ? a : zero;
            else gf[c - 2] = a;
        }
#pragma unroll
        for (int g = 0; g < kCiCh * kCiIn / 16; ++g) {                      // w1[o][c]: d1[o] * x[c]
            f2 sums[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) sums[i] = f2_mul(d1[(g * 16 + i) / kCiIn], x[0][(g * 16 + i) % kCiIn]);
            reduce_group(sums, [g](int i) { return kCiW1 + g * 16 + i; });
        }
        {
            f2 sums[16];                                                    // b1: d1;  b3: go;  d/d(ref): dx of the two rel inputs
#pragma unroll
            for (int i = 0; i < 16; ++i) sums[i] = i < 8 ? d1[i < 8 ? i : 0] : i == 8 ? go : i < 11 ? dx01[i == 10 ? 1 : 0] : zero;
            reduce_group(sums, [](int i) { return i < 8 ? kCiB1 + i : i == 8 ? kCiB3 : i < 11 ? kCiParams + (i - 9) : -1; });
        }
    }
#pragma unroll
    for (int c = 0; c < kCiFeat; ++c) {
        if constexpr (DET) {
            float *dst = feat_part + (((size_t)blockIdx.y * gridDim.z + b) * kCiFeat + c) * HW;
            if (live0) dst[pa] = f2_lo(gf[c]);
            if (live1) dst[pb] = f2_hi(gf[c]);
            continue;
        }
        float *dst = grad_feats + ((size_t)b * kCiFeat + c) * HW;
        if (live0) atomicAdd(dst + pa, f2_lo(gf[c]));
        if (live1) atomicAdd(dst + pb, f2_hi(gf[c]));
    }
}

// Fixed-order reduction of condinst_bwd<true>'s partials.  Threads [0, N*8*HW) sum the feature partials of the instance
// chunks image b actually has, in chunk order; threads [N*8*HW, + I*171) sum the per-instance partials over the warp slots
// in slot order.  Every output element is written.
__global__ void __launch_bounds__(256)
condinst_bwd_reduce(const float *__restrict__ feat_part, const float *__restrict__ sum_part, const int *__restrict__ inst_start,
                    int N, int HW, int I, int nslots, float *__restrict__ grad_feats, float *__restrict__ grad_params,
                    float *__restrict__ grad_refs)
{
    const long long nf = (long long)N * kCiFeat * HW, ns = (long long)I * kCiSums;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < nf + ns; t += (long long)gridDim.x * blockDim.x) {
        float acc = 0.f;
        if (t < nf) {
            const int b = (int)(t / ((long long)kCiFeat * HW));
            const int chunks = (inst_start[b + 1] - inst_start[b] + kCiChunk - 1) / kCiChunk;
            for (int y = 0; y < chunks; ++y) acc += feat_part[(size_t)y * nf + t];
            grad_feats[t] = acc;
        } else {
            const long long u = t - nf;
            for (int sl = 0; sl < nslots; ++sl) acc += sum_part[(size_t)sl * ns + u];
            const int i = (int)(u / kCiSums), j = (int)(u % kCiSums);
            if (j < kCiParams) grad_params[(size_t)i * kCiParams + j] = acc;
            else grad_refs[(size_t)i * 2 + (j - kCiParams)] = acc;
        }
    }
}

// ---- aligned_bilinear (ddetrs.py:921-942): out[Y, X] of size (f*h, f*w) samples the replicate-padded input at
// ((Y - f/2)^+ / f, (X - f/2)^+ / f) with align_corners weights.  src index pair + fraction for one output coordinate:
__device__ __forceinline__ void ab_src(int o, int f, int n, int &i0, int &i1, float &fr) {
    const int p = max(o - f / 2, 0);
    i0 = p / f;
    fr = (float)(p - i0 * f) / (float)f;
    i1 = min(i0 + 1, n - 1);
}

constexpr int kAbRows = 16;                 // output rows (forward) / input rows (backward) per block

// grid: (planes, row tiles).  F = compile-time factor (0: use the run-time f).  VEC = 4 needs (f * w) % 4 == 0.
template <int F, int VEC>
__global__ void __launch_bounds__(256)
aligned_bilinear_fwd(const float *__restrict__ in, int h, int w, int f_rt, float *__restrict__ out) {
    const int f = F ? F : f_rt;
    const int oh = h * f, ow = w * f, owv = ow / VEC;
    const float *src = in + (size_t)blockIdx.x * h * w;
    float *dst = out + (size_t)blockIdx.x * oh * ow;
    const int Y0 = blockIdx.y * kAbRows, rows = min(kAbRows, oh - Y0);
    for (int t = threadIdx.x; t < rows * owv; t += 256) {
        const int r = t / owv, Y = Y0 + r, X0 = (t - r * owv) * VEC;
        int y0, y1; float fy;
        ab_src(Y, f, h, y0, y1, fy);
        const float *top = src + (size_t)y0 * w, *bot = src + (size_t)y1 * w;
        float o[VEC];
#pragma unroll
        for (int q = 0; q < VEC; ++q) {
            int x0, x1; float fx;
            ab_src(X0 + q, f, w, x0, x1, fx);
            const float a = (1.f - fx) * __ldg(top + x0) + fx * __ldg(top + x1);
            const float c = (1.f - fx) * __ldg(bot + x0) + fx * __ldg(bot + x1);
            o[q] = (1.f - fy) * a + fy * c;
        }
        if (VEC == 4) *reinterpret_cast<float4 *>(dst + (size_t)Y * ow + X0) = make_float4(o[0], o[1 % VEC], o[2 % VEC], o[3 % VEC]);
        else dst[(size_t)Y * ow + X0] = o[0];
    }
}

// gather form of the transpose: input pixel (y, x) collects from every output whose source pair contains it -- source
// positions in [y - 1, y + 1), i.e. Y in [f*(y-1) + f/2, f*(y+1) + f/2), plus the clamped head [0, f/2) for y == 0.
template <int F>
__global__ void __launch_bounds__(256)
aligned_bilinear_bwd(const float *__restrict__ gout, int h, int w, int f_rt, float *__restrict__ gin) {
    const int f = F ? F : f_rt;
    const int oh = h * f, ow = w * f;
    const float *g = gout + (size_t)blockIdx.x * oh * ow;
    float *dst = gin + (size_t)blockIdx.x * h * w;
    const int y0b = blockIdx.y * kAbRows, rows = min(kAbRows, h - y0b);
    for (int t = threadIdx.x; t < rows * w; t += 256) {
        const int r = t / w, y = y0b + r, x = t - r * w;
        const int Ya = y == 0 ? 0 : max(0, f * (y - 1) + f / 2), Yb = min(oh, f * (y + 1) + f / 2);
        const int Xa = x == 0 ? 0 : max(0, f * (x - 1) + f / 2), Xb = min(ow, f * (x + 1) + f / 2);
        float acc = 0.f;
        for (int Y = Ya; Y < Yb; ++Y) {
            int s0, s1; float fy;
            ab_src(Y, f, h, s0, s1, fy);
            const float wy = (s0 == y ? 1.f - fy : 0.f) + (s1 == y ? fy : 0.f);
            if (wy == 0.f) continue;
            float row = 0.f;
            for (int X = Xa; X < Xb; ++X) {
                int x0, x1; float fx;
                ab_src(X, f, w, x0, x1, fx);
                const float wx = (x0 == x ? 1.f - fx : 0.f) + (x1 == x ? fx : 0.f);
                row = fmaf(wx, __ldg(g + (size_t)Y * ow + X), row);
            }
            acc = fmaf(wy, row, acc);
        }
        dst[t + (size_t)y0b * w] = acc;
    }
}

// ---- factor 2 (mask_feat_stride 8 -> mask_out_stride 4, every UNINEXT config), closed form, w even:
//   out[Y]: Y == 0 -> in[0];  Y odd -> in[(Y - 1) / 2];  Y even -> (in[Y/2 - 1] + in[Y/2]) / 2         (same along X)
//   transpose: gin[y] = (y == 0 ? 1 : 1/2) g[2y] + g[2y + 1] + 1/2 g[2y + 2]                            (last term absent for y == h - 1)
// grid: (planes, row tiles); four outputs (forward) / two inputs (backward) per thread-iteration.
__global__ void __launch_bounds__(256)
aligned_bilinear2_fwd(const float *__restrict__ in, int h, int w, float *__restrict__ out) {
    const int oh = 2 * h, ow = 2 * w, owv = ow / 4;
    const float *src = in + (size_t)blockIdx.x * h * w;
    float *dst = out + (size_t)blockIdx.x * oh * ow;
    const int Y0 = blockIdx.y * kAbRows, rows = min(kAbRows, oh - Y0);
    // thread -> (column group, first row): one division per thread, none per element
    const int per = min(owv, 256), rstep = 256 / per, cg0 = threadIdx.x % per, r0 = threadIdx.x / per;
    if (r0 >= rstep) return;
    for (int cg = cg0; cg < owv; cg += per) {
        const int X0 = cg * 4, c = X0 >> 1, cm = max(c - 1, 0);
        for (int r = r0; r < rows; r += rstep) {
            const int Y = Y0 + r, p = max(Y - 1, 0), y0 = p >> 1;
            const bool two = (p & 1) != 0;
            const float *ra = src + (size_t)y0 * w, *rb = src + (size_t)min(y0 + 1, h - 1) * w;
            float a = __ldg(ra + cm), b = __ldg(ra + c), d = __ldg(ra + c + 1);
            float o0 = X0 == 0 ? b : 0.5f * a + 0.5f * b, o1 = b, o2 = 0.5f * b + 0.5f * d, o3 = d;
            if (two) {
                a = __ldg(rb + cm); b = __ldg(rb + c); d = __ldg(rb + c + 1);
                o0 = 0.5f * o0 + 0.5f * (X0 == 0 ? b : 0.5f * a + 0.5f * b);
                o1 = 0.5f * o1 + 0.5f * b;
                o2 = 0.5f * o2 + 0.5f * (0.5f * b + 0.5f * d);
                o3 = 0.5f * o3 + 0.5f * d;
            }
            *reinterpret_cast<float4 *>(dst + (size_t)Y * ow + X0) = make_float4(o0, o1, o2, o3);
        }
    }
}

__global__ void __launch_bounds__(256)
aligned_bilinear2_bwd(const float *__restrict__ gout, int h, int w, float *__restrict__ gin) {
    const int oh = 2 * h, ow = 2 * w, wv = w / 2;
    const float *g = gout + (size_t)blockIdx.x * oh * ow;
    float *dst = gin + (size_t)blockIdx.x * h * w;
    const int y0b = blockIdx.y * kAbRows, rows = min(kAbRows, h - y0b);
    const int per = min(wv, 256), rstep = 256 / per, cg0 = threadIdx.x % per, r0 = threadIdx.x / per;
    if (r0 >= rstep) return;
    for (int cg = cg0; cg < wv; cg += per) {
        const int x = cg * 2;
        const float wx0 = x == 0 ? 1.f : 0.5f;
        const bool tail = 2 * x + 4 < ow;
        for (int r = r0; r < rows; r += rstep) {
            const int y = y0b + r;
            float s0 = 0.f, s1 = 0.f;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const int Y = 2 * y + k;
                if (Y >= oh) break;
                const float wy = k == 1 ? 1.f : (k == 0 && y > 0) || k == 2 ? 0.5f : 1.f;
                const float4 v = __ldg(reinterpret_cast<const float4 *>(g + (size_t)Y * ow + 2 * x));
                const float e = tail ? __ldg(g + (size_t)Y * ow + 2 * x + 4) : 0.f;
                s0 = fmaf(wy, wx0 * v.x + v.y + 0.5f * v.z, s0);
                s1 = fmaf(wy, 0.5f * v.z + v.w + 0.5f * e, s1);
            }
            *reinterpret_cast<float2 *>(dst + (size_t)y * w + x) = make_float2(s0, s1);
        }
    }
}

}  // namespace msda
