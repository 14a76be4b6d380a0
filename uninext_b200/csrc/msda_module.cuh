// msda_module.cuh -- memory-bound kernels for the CALLERS of the op (SURVEY.md section 8 rows f-1 / f-2):
//   * sampling prologue: raw projection [rows, M*L*P*3] -> softmax(attention logits) + sampling-location arithmetic,
//     written directly in the op's layouts (reference: ops/modules/ms_deform_attn.py:99-112, five elementwise passes);
//   * its backward (softmax backward + location scaling) producing the gradient of the raw projection;
//   * column sums (bias gradients of the bracketing Linears);
//   * residual-add + LayerNorm forward / backward (deformable_transformer.py:354-356,359 `norm(src + dropout(x))`).
// All fp32; every kernel is one pass over its operands.
#pragma once

#include "msda_common.cuh"

namespace msda {

template <int G>
__device__ __forceinline__ float group_max(float v) {
#pragma unroll
    for (int d = G / 2; d >= 1; d >>= 1) v = fmaxf(v, __shfl_xor_sync(kFullMask, v, d, G));
    return v;
}
template <int G>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
    for (int d = G / 2; d >= 1; d >>= 1) v += __shfl_xor_sync(kFullMask, v, d, G);
    return v;
}

// proj row layout (one GEMM over the concatenated sampling_offsets / attention_weights Linears):
//   [0, M*LP*2)          offsets, ordered (m, l, p, xy)   -- ms_deform_attn.py:99
//   [M*LP*2, M*LP*3)     attention logits, ordered (m, l*p) -- ms_deform_attn.py:100
// One lane per tap, G = pow2 >= L*P lanes per (row, head).
template <int G>
__global__ void __launch_bounds__(256)
msda_prologue_fwd(const float *__restrict__ proj, const float *__restrict__ ref, const int64_t *__restrict__ shapes,
                  long long npairs, int M, int L, int P, int refdim, float *__restrict__ loc, float *__restrict__ attn)
{
    const int LP = L * P, ncols = M * LP * 3;
    const long long gid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) / G;
    const int j = threadIdx.x % G;
    const bool live = gid < npairs;
    const long long pair = live ? gid : npairs - 1;
    const long long r = pair / M;
    const int m = (int)(pair % M);
    const bool tap = j < LP;
    const float *row = proj + r * ncols;
    const float logit = tap ? __ldg(row + M * LP * 2 + m * LP + j) : -INFINITY;
    const float mx = group_max<G>(logit);
    const float e = tap ? expf(logit - mx) : 0.f;
    const float a = e / group_sum<G>(e);                                    // F.softmax(..., -1), ms_deform_attn.py:101
    if (!(tap && live)) return;
    const float2 off = make_float2(__ldg(row + 2 * (m * LP + j)), __ldg(row + 2 * (m * LP + j) + 1));   // rows may be 4-byte aligned only
    const int l = j / P;
    const float *rp = ref + (r * L + l) * refdim;
    float2 o;
    if (refdim == 2) {                                                      // ms_deform_attn.py:103-106
        o.x = __ldg(rp) + off.x / (float)shapes[2 * l + 1];
        o.y = __ldg(rp + 1) + off.y / (float)shapes[2 * l];
    } else {                                                                // ms_deform_attn.py:107-109
        o.x = __ldg(rp) + off.x / (float)P * __ldg(rp + 2) * 0.5f;
        o.y = __ldg(rp + 1) + off.y / (float)P * __ldg(rp + 3) * 0.5f;
    }
    reinterpret_cast<float2 *>(loc)[pair * LP + j] = o;
    attn[pair * LP + j] = a;
}

// grad wrt the raw projection.  d logits = a * (ga - sum(a * ga));  d offsets = gl * d(loc)/d(off).
template <int G>
__global__ void __launch_bounds__(256)
msda_prologue_bwd(const float *__restrict__ grad_loc, const float *__restrict__ grad_attn, const float *__restrict__ attn,
                  const float *__restrict__ ref, const int64_t *__restrict__ shapes, long long npairs, int M, int L,
                  int P, int refdim, float *__restrict__ grad_proj)
{
    const int LP = L * P, ncols = M * LP * 3;
    const long long gid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) / G;
    const int j = threadIdx.x % G;
    const bool live = gid < npairs;
    const long long pair = live ? gid : npairs - 1;
    const long long r = pair / M;
    const int m = (int)(pair % M);
    const bool tap = j < LP;
    const float a = tap ? __ldg(attn + pair * LP + j) : 0.f;
    const float ga = tap ? __ldg(grad_attn + pair * LP + j) : 0.f;
    const float dot = group_sum<G>(a * ga);
    if (!(tap && live)) return;
    float *row = grad_proj + r * ncols;
    row[M * LP * 2 + m * LP + j] = a * (ga - dot);
    const float2 gl = __ldg(reinterpret_cast<const float2 *>(grad_loc) + pair * LP + j);
    const int l = j / P;
    float2 g;
    if (refdim == 2) {
        g.x = gl.x / (float)shapes[2 * l + 1];
        g.y = gl.y / (float)shapes[2 * l];
    } else {
        const float *rp = ref + (r * L + l) * refdim;
        g.x = gl.x * (__ldg(rp + 2) * 0.5f / (float)P);
        g.y = gl.y * (__ldg(rp + 3) * 0.5f / (float)P);
    }
    row[2 * (m * LP + j)] = g.x;
    row[2 * (m * LP + j) + 1] = g.y;
}

// Deterministic variants (DET = true) of the column sums below: the CTA's partial row, already summed in a fixed order,
// is stored to row blockIdx.x of a [gridDim.x, cols] scratch instead of being added to the result with a float red;
// msda_sum_partials then adds the rows in index order.
__device__ __forceinline__ void colsum_out(bool det, float *out, int cols, int c, float4 acc) {
    if (det) reinterpret_cast<float4 *>(out + (size_t)blockIdx.x * cols)[c] = acc;
    else red_add_v4(out + 4 * c, acc.x, acc.y, acc.z, acc.w);
}

// out[c] = sum_p part[p, c] for p = 0 .. nparts-1 in order.
__global__ void __launch_bounds__(256)
msda_sum_partials(const float *__restrict__ part, int nparts, int cols, float *__restrict__ out)
{
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < cols; c += gridDim.x * blockDim.x) {
        float acc = 0.f;
        for (int p = 0; p < nparts; ++p) acc += part[(size_t)p * cols + c];
        out[c] = acc;
    }
}

// out[c] += sum over this CTA's rows of x[r, c].  `out` must be zero on entry.  Thread (rl, c) sums the float4 column slice
// c over rows r0+rl, r0+rl+RL, ...; the RL row-lanes are then combined in shared memory and leave as one 16-byte red.
template <bool DET = false>
__global__ void __launch_bounds__(256)
msda_colsum(const float *__restrict__ x, long long rows, int cols, int rows_per_cta, float *__restrict__ out)
{
    __shared__ float4 part[256];
    const long long r0 = (long long)blockIdx.x * rows_per_cta;
    const long long r1 = min(rows, r0 + rows_per_cta);
    const int c4 = cols / 4;
    const int cs = min(c4, (int)blockDim.x);          // column slices handled per sweep
    const int RL = blockDim.x / cs;                    // row lanes
    const int ct = threadIdx.x % cs, rl = threadIdx.x / cs;
    for (int cb = 0; cb < c4; cb += cs) {              // uniform trip count: the loop body holds block barriers
        const int c = cb + ct;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        if (rl < RL && c < c4) {
            const float4 *p = reinterpret_cast<const float4 *>(x) + (r0 + rl) * c4 + c;
#pragma unroll 8
            for (long long r = r0 + rl; r < r1; r += RL, p += (long long)RL * c4) {
                const float4 v = __ldg(p);
                acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
            }
        }
        part[threadIdx.x] = acc;
        __syncthreads();
        if (rl == 0 && c < c4) {
            for (int k = 1; k < RL; ++k) {
                const float4 t = part[k * cs + ct];
                acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w;
            }
            colsum_out(DET, out, cols, c, acc);
        }
        __syncthreads();
    }
}

// ReLU backward fused with the bias gradient of the Linear in front of it (FFN linear1, deformable_transformer.py:345-349):
//   g2[r, c] = y[r, c] > 0 ? g[r, c] : 0 ;   out[c] += sum_r g2[r, c]
// One pass over g and y instead of threshold_backward followed by a separate column-sum read of g2 (366 MB at cfg2).
template <bool DET = false>
__global__ void __launch_bounds__(256)
msda_relu_bwd_colsum(const float *__restrict__ g, const float *__restrict__ y, long long rows, int cols, int rows_per_cta,
                     float *__restrict__ g2, float *__restrict__ out)
{
    __shared__ float4 part[256];
    const long long r0 = (long long)blockIdx.x * rows_per_cta;
    const long long r1 = min(rows, r0 + rows_per_cta);
    const int c4 = cols / 4;
    const int cs = min(c4, (int)blockDim.x);
    const int RL = blockDim.x / cs;
    const int ct = threadIdx.x % cs, rl = threadIdx.x / cs;
    for (int cb = 0; cb < c4; cb += cs) {
        const int c = cb + ct;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        if (rl < RL && c < c4) {
            long long i = (r0 + rl) * c4 + c;
#pragma unroll 4
            for (long long r = r0 + rl; r < r1; r += RL, i += (long long)RL * c4) {
                const float4 gv = __ldg(reinterpret_cast<const float4 *>(g) + i);
                const float4 yv = __ldg(reinterpret_cast<const float4 *>(y) + i);
                const float4 o = make_float4(yv.x > 0.f ? gv.x : 0.f, yv.y > 0.f ? gv.y : 0.f, yv.z > 0.f ? gv.z : 0.f,
                                             yv.w > 0.f ? gv.w : 0.f);
                reinterpret_cast<float4 *>(g2)[i] = o;
                acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w;
            }
        }
        part[threadIdx.x] = acc;
        __syncthreads();
        if (rl == 0 && c < c4) {
            for (int k = 1; k < RL; ++k) {
                const float4 t = part[k * cs + ct];
                acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w;
            }
            colsum_out(DET, out, cols, c, acc);
        }
        __syncthreads();
    }
}

// ---- geometry feeding the op (SURVEY.md section 8 f-3; deformable_transformer_dino.py:132-171,289-301,612-646) -----------------
// The reference builds these with ~20 small PyTorch kernels per forward (meshgrid / linspace / cat / stack per level, with a
// device->host sync for every level shape).  Here: one launch each, level table read on the device.

// counts[n, l] = (valid_W, valid_H): un-padded extent of level l in image n, from the flattened padding mask
// (get_valid_ratio, _dino.py:164-171: first row / first column of the level's mask).  One warp per (n, l).
__global__ void __launch_bounds__(256)
msda_valid_counts(const unsigned char *__restrict__ mask, const int64_t *__restrict__ shapes, const int64_t *__restrict__ lsi,
                  int N, int S, int L, int *__restrict__ counts)
{
    const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (gw >= N * L) return;
    const int n = gw / L, l = gw - n * L;
    const int H = (int)shapes[2 * l], W = (int)shapes[2 * l + 1];
    const unsigned char *m = mask + (size_t)n * S + (int)lsi[l];
    int vw = 0, vh = 0;
    for (int x = lane; x < W; x += 32) vw += m[x] == 0;                 // ~mask[:, 0, :]
    for (int y = lane; y < H; y += 32) vh += m[(size_t)y * W] == 0;     // ~mask[:, :, 0]
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) { vw += __shfl_xor_sync(kFullMask, vw, d); vh += __shfl_xor_sync(kFullMask, vh, d); }
    if (lane == 0) { counts[2 * gw] = vw; counts[2 * gw + 1] = vh; }
}

__device__ __forceinline__ int level_of(const int64_t *lsi, const int64_t *shapes, int L, int s, int &x, int &y, int &H, int &W) {
    int l = 0;
    while (l + 1 < L && s >= (int)lsi[l + 1]) ++l;
    H = (int)shapes[2 * l]; W = (int)shapes[2 * l + 1];
    const int p = s - (int)lsi[l];
    y = p / W; x = p - y * W;
    return l;
}

// ref[n, s, l, :] = ((x + 0.5) / (vr[n, ls, 0] * W), (y + 0.5) / (vr[n, ls, 1] * H)) * vr[n, l, :]   (_dino.py:289-301), ls = level of s
__global__ void __launch_bounds__(256)
msda_encoder_ref_points(const float *__restrict__ vr, const int64_t *__restrict__ shapes, const int64_t *__restrict__ lsi,
                        int N, int S, int L, float *__restrict__ ref)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)N * S) return;
    const int n = (int)(t / S), s = (int)(t - (long long)n * S);
    int x, y, H, W;
    const int ls = level_of(lsi, shapes, L, s, x, y, H, W);
    const float *v = vr + (size_t)n * L * 2;
    const float rx = ((float)x + 0.5f) / (v[2 * ls] * (float)W), ry = ((float)y + 0.5f) / (v[2 * ls + 1] * (float)H);
    float2 *o = reinterpret_cast<float2 *>(ref) + (size_t)t * L;
    for (int l = 0; l < L; ++l) o[l] = make_float2(rx * v[2 * l], ry * v[2 * l + 1]);
}

// Two-stage proposals (_dino.py:132-156): prop = logit((x+.5)/valid_W, (y+.5)/valid_H, 0.05*2^l, 0.05*2^l), +inf where the
// position is padded or any coordinate is outside (0.01, 0.99); keep = position survives.
__global__ void __launch_bounds__(256)
msda_encoder_proposals(const unsigned char *__restrict__ mask, const int *__restrict__ counts, const int64_t *__restrict__ shapes,
                       const int64_t *__restrict__ lsi, int N, int S, int L, float base_scale, float *__restrict__ prop,
                       unsigned char *__restrict__ keep)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)N * S) return;
    const int n = (int)(t / S), s = (int)(t - (long long)n * S);
    int x, y, H, W;
    const int l = level_of(lsi, shapes, L, s, x, y, H, W);
    const int *c = counts + ((size_t)n * L + l) * 2;
    const float wh = base_scale * (float)(1 << l);
    const float p[4] = {((float)x + 0.5f) / (float)c[0], ((float)y + 0.5f) / (float)c[1], wh, wh};
    bool ok = mask[t] == 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) ok = ok && p[i] > 0.01f && p[i] < 0.99f;
    float4 o;
    const float inf = __int_as_float(0x7f800000);
    o.x = ok ? logf(p[0] / (1.f - p[0])) : inf; o.y = ok ? logf(p[1] / (1.f - p[1])) : inf;
    o.z = ok ? logf(p[2] / (1.f - p[2])) : inf; o.w = ok ? logf(p[3] / (1.f - p[3])) : inf;
    reinterpret_cast<float4 *>(prop)[t] = o;
    keep[t] = ok ? 1 : 0;
}

// Sine position embedding of box coordinates (get_sine_pos_embed, _dino.py:612-646): out[r, slot(k) * F + j] =
// sin / cos (j even / odd) of pos[r, k] * 2 pi / T^(2 (j / 2) / F); slot swaps components 0 and 1 when exchange_xy.
// BWD: grad_pos[r, k] = sum_j g * d/dpos (one warp per (r, k)).
template <bool BWD>
__global__ void __launch_bounds__(256)
msda_sine_pos_embed(const float *__restrict__ pos, const float *__restrict__ gout, long long R, int n, int F, float temperature,
                    int exchange_xy, float *__restrict__ out)
{
    const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (gw >= R * n) return;
    const long long r = gw / n;
    const int k = (int)(gw - r * n);
    const int slot = (exchange_xy && n >= 2 && k < 2) ? 1 - k : k;
    const float p = pos[gw] * 6.283185307179586f;
    float acc = 0.f;
    for (int j = lane; j < F; j += 32) {
        const float dim_t = powf(temperature, (float)(2 * (j / 2)) / (float)F);
        const float a = p / dim_t;
        if (!BWD) {
            out[(r * n + slot) * F + j] = (j & 1) ? cosf(a) : sinf(a);
        } else {
            const float g = gout[(r * n + slot) * F + j];
            acc += g * ((j & 1) ? -sinf(a) : cosf(a)) * (6.283185307179586f / dim_t);
        }
    }
    if (BWD) {
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) acc += __shfl_xor_sync(kFullMask, acc, d);
        if (lane == 0) out[gw] = acc;
    }
}

// z = a + b (b may be null);  y = (z - mean) * rstd * gamma + beta, one warp per row of C = 128*V channels.
template <int V>
__global__ void __launch_bounds__(256)
msda_add_layernorm_fwd(const float *__restrict__ a, const float *__restrict__ b, const float *__restrict__ gamma,
                       const float *__restrict__ beta, long long rows, float eps, float *__restrict__ z,
                       float *__restrict__ y, float *__restrict__ mean, float *__restrict__ rstd)
{
    constexpr int C = 128 * V;
    const int lane = threadIdx.x & 31;
    const long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= rows) return;
    float4 v[V];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < V; ++i) {
        const long long o = row * (C / 4) + i * 32 + lane;
        v[i] = __ldg(reinterpret_cast<const float4 *>(a) + o);
        if (b != nullptr) {
            const float4 t = __ldg(reinterpret_cast<const float4 *>(b) + o);
            v[i].x += t.x; v[i].y += t.y; v[i].z += t.z; v[i].w += t.w;
        }
        s += v[i].x + v[i].y + v[i].z + v[i].w;
    }
    const float mu = group_sum<32>(s) * (1.f / C);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < V; ++i) {
        const float dx = v[i].x - mu, dy = v[i].y - mu, dz = v[i].z - mu, dw = v[i].w - mu;
        q += dx * dx + dy * dy + dz * dz + dw * dw;
    }
    const float rs = rsqrtf(group_sum<32>(q) * (1.f / C) + eps);
#pragma unroll
    for (int i = 0; i < V; ++i) {
        const long long o = row * (C / 4) + i * 32 + lane;
        const float4 g = __ldg(reinterpret_cast<const float4 *>(gamma) + i * 32 + lane);
        const float4 bt = __ldg(reinterpret_cast<const float4 *>(beta) + i * 32 + lane);
        if (z != nullptr) reinterpret_cast<float4 *>(z)[o] = v[i];
        reinterpret_cast<float4 *>(y)[o] = make_float4((v[i].x - mu) * rs * g.x + bt.x, (v[i].y - mu) * rs * g.y + bt.y,
                                                       (v[i].z - mu) * rs * g.z + bt.z, (v[i].w - mu) * rs * g.w + bt.w);
    }
    if (lane == 0) { mean[row] = mu; rstd[row] = rs; }
}

// dz = rstd * (dy*gamma - mean(dy*gamma) - xhat * mean(dy*gamma*xhat));  dgamma += sum_rows dy*xhat;  dbeta += sum_rows dy.
// Each warp walks rows warp, warp+W, ...; its per-lane column partials are combined across the CTA's warps in shared
// memory and leave the CTA as one 16-byte red per lane-slice.  dgamma / dbeta must be zero on entry.
// DET: dgamma / dbeta are [gridDim.x, cols] scratch rows instead (see colsum_out).
template <int V, bool DET = false>
__global__ void __launch_bounds__(256)
msda_layernorm_bwd(const float *__restrict__ dy, const float *__restrict__ z, const float *__restrict__ gamma,
                   const float *__restrict__ mean, const float *__restrict__ rstd, long long rows, int rows_per_cta,
                   float *__restrict__ dz, float *__restrict__ dgamma, float *__restrict__ dbeta)
{
    constexpr int C = 128 * V;
    __shared__ float4 sg[8][V * 32], sb[8][V * 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long r0 = (long long)blockIdx.x * rows_per_cta, r1 = min(rows, r0 + rows_per_cta);
    float4 g[V], ag[V], ab[V];
#pragma unroll
    for (int i = 0; i < V; ++i) {
        g[i] = __ldg(reinterpret_cast<const float4 *>(gamma) + i * 32 + lane);
        ag[i] = ab[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    for (long long row = r0 + warp; row < r1; row += 8) {
        const float mu = __ldg(mean + row), rs = __ldg(rstd + row);
        float4 d[V], xh[V];
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int i = 0; i < V; ++i) {
            const long long o = row * (C / 4) + i * 32 + lane;
            d[i] = __ldg(reinterpret_cast<const float4 *>(dy) + o);
            const float4 zz = __ldg(reinterpret_cast<const float4 *>(z) + o);
            xh[i] = make_float4((zz.x - mu) * rs, (zz.y - mu) * rs, (zz.z - mu) * rs, (zz.w - mu) * rs);
            ab[i].x += d[i].x; ab[i].y += d[i].y; ab[i].z += d[i].z; ab[i].w += d[i].w;
            ag[i].x += d[i].x * xh[i].x; ag[i].y += d[i].y * xh[i].y; ag[i].z += d[i].z * xh[i].z; ag[i].w += d[i].w * xh[i].w;
            d[i].x *= g[i].x; d[i].y *= g[i].y; d[i].z *= g[i].z; d[i].w *= g[i].w;       // dy * gamma
            s1 += d[i].x + d[i].y + d[i].z + d[i].w;
            s2 += d[i].x * xh[i].x + d[i].y * xh[i].y + d[i].z * xh[i].z + d[i].w * xh[i].w;
        }
        s1 = group_sum<32>(s1) * (1.f / C);
        s2 = group_sum<32>(s2) * (1.f / C);
#pragma unroll
        for (int i = 0; i < V; ++i) {
            const long long o = row * (C / 4) + i * 32 + lane;
            reinterpret_cast<float4 *>(dz)[o] = make_float4(rs * (d[i].x - s1 - xh[i].x * s2), rs * (d[i].y - s1 - xh[i].y * s2),
                                                            rs * (d[i].z - s1 - xh[i].z * s2), rs * (d[i].w - s1 - xh[i].w * s2));
        }
    }
#pragma unroll
    for (int i = 0; i < V; ++i) { sg[warp][i * 32 + lane] = ag[i]; sb[warp][i * 32 + lane] = ab[i]; }
    __syncthreads();
    for (int c = threadIdx.x; c < V * 32; c += blockDim.x) {
        float4 tg = sg[0][c], tb = sb[0][c];
#pragma unroll
        for (int w = 1; w < 8; ++w) {
            tg.x += sg[w][c].x; tg.y += sg[w][c].y; tg.z += sg[w][c].z; tg.w += sg[w][c].w;
            tb.x += sb[w][c].x; tb.y += sb[w][c].y; tb.z += sb[w][c].z; tb.w += sb[w][c].w;
        }
        colsum_out(DET, dgamma, C, c, tg);
        colsum_out(DET, dbeta, C, c, tb);
    }
}

}  // namespace msda
