// msda_common.cuh -- shared device helpers for the sm_100a multi-scale deformable attention kernels.
//
// Semantics follow the reference kernels in
//   /root/reference/projects/UNINEXT/uninext/models/deformable_detr/ops/src/cuda/ms_deform_im2col_cuda.cuh ("cuh"):
//   pixel mapping cuh:285-286, validity window cuh:288, per-corner predicates cuh:56-78, weights cuh:80-83,
//   gradients cuh:112-158.  Nothing here is derived from that file's code structure: a tap is resolved ONCE by one
//   lane into (clamped row indices, masked corner weights) and shared with the lanes that own the channels.
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace msda {

constexpr int kMaxLevels = 8;         // level table kept in shared memory by the tiled kernels
constexpr unsigned kFullMask = 0xffffffffu;

// ---- programmatic dependent launch (PDL) --------------------------------------------------------------------------
// grad_value must be zero before the backward kernel's first red.  With MSDA_KNOB_ZERO_FILL = 2 the zero-fill kernel
// below and the backward kernel are a PDL pair: the fill kernel lets its dependent launch as soon as all of its CTAs are
// running, the backward kernel builds its work map, initialises its mbarriers and starts its first TMA tap loads (none
// of which touch grad_value), and only then waits for the fill to have completed and flushed.  Without the launch
// attribute both instructions are no-ops.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait_primary() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// Zero-fill of a 16-byte aligned buffer of n16 x 16 bytes: one wave of CTAs, 16-byte stores, grid stride.
__global__ void __launch_bounds__(256) msda_zero_fill(uint4 *__restrict__ p, unsigned long long n16) {
    pdl_launch_dependents();
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    const uint4 z = make_uint4(0u, 0u, 0u, 0u);
    unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
#pragma unroll 4
    for (; i < n16; i += stride) p[i] = z;
}

// Geometry of one bilinear tap, resolved against one level map.
//   r0 / r1 : row index (within one batch element, i.e. in [0, S)) of the clamped (h0, w0) / (h1, w0) corners.
//             Clamping keeps every address legal; corners outside the map get weight 0 through `mask`.
//   dw      : 1 when the clamped w1 differs from the clamped w0 (i.e. the right-hand corners are one row further).
//   mask    : bit k set <=> corner k (00, 01, 10, 11) lies inside the map AND the tap passes the window test.
struct TapGeom {
    float lh, lw;
    int r0, r1;
    int dw;
    unsigned mask;
};

__device__ __forceinline__ TapGeom tap_geometry(float x, float y, int H, int W, int start) {
    TapGeom g;
    // Same rounding sequence as the reference: product rounded to fp32, then the 0.5 shift (cuh:285-286).
    const float h_im = __fadd_rn(__fmul_rn(y, (float)H), -0.5f);
    const float w_im = __fadd_rn(__fmul_rn(x, (float)W), -0.5f);
    const bool inside = (h_im > -1.f) && (w_im > -1.f) && (h_im < (float)H) && (w_im < (float)W);   // cuh:288
    const float hf = floorf(h_im), wf = floorf(w_im);
    g.lh = h_im - hf;
    g.lw = w_im - wf;
    int h0 = inside ? (int)hf : 0;
    int w0 = inside ? (int)wf : 0;
    const int h1 = h0 + 1, w1 = w0 + 1;
    unsigned m = 0;
    if (inside) {
        const bool t = h0 >= 0, b = h1 <= H - 1, l = w0 >= 0, r = w1 <= W - 1;     // cuh:56,62,68,74
        m = (unsigned)(t && l) | ((unsigned)(t && r) << 1) | ((unsigned)(b && l) << 2) | ((unsigned)(b && r) << 3);
    }
    g.mask = m;
    const int ch0 = max(h0, 0), ch1 = min(h1, H - 1), cw0 = max(w0, 0), cw1 = min(w1, W - 1);
    g.r0 = start + ch0 * W + cw0;
    g.r1 = start + ch1 * W + cw0;
    g.dw = cw1 - cw0;
    return g;
}

// Masked corner weights of a tap with attention weight a (corner k outside the map or window: 0).
__device__ __forceinline__ float4 masked_weights(const TapGeom &g, float a) {
    const float hh = 1.f - g.lh, hw = 1.f - g.lw;
    return make_float4((g.mask & 1u) ? hh * hw * a : 0.f, (g.mask & 2u) ? hh * g.lw * a : 0.f,
                       (g.mask & 4u) ? g.lh * hw * a : 0.f, (g.mask & 8u) ? g.lh * g.lw * a : 0.f);
}

// Vector access to one slice of a value / grad row, widened to fp32 registers.  VEC = elements per lane:
// fp32: 4 (16 bytes); bf16: 8 (16 bytes, forward) or 4 (8 bytes, backward -- keeps one lane's grad_value slice a
// contiguous 16-byte fp32 quad so that every red.v4 fills whole sectors).
template <typename T, int VEC> struct RowVec;

template <> struct RowVec<float, 4> {
    static constexpr int kElems = 4;
    __device__ static __forceinline__ void load(const float *p, float (&v)[4]) {
        const float4 t = __ldg(reinterpret_cast<const float4 *>(p));
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    }
    __device__ static __forceinline__ void store(float *p, const float (&v)[4]) {
        *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
    }
};

// fp32, 8 channels per lane: one 32-byte access (sm_100 LDG.256 / STG.256 would need 32-byte alignment of the tensor, which
// the router checks).  4 lanes cover a 128-byte row, 8 rows per warp instruction: 119 B/clk/SM from L1 against 80 for the
// 16-byte shape (profiles/r02b_ubench_smem_rmw_and_egress.txt).
template <> struct RowVec<float, 8> {
    static constexpr int kElems = 8;
    __device__ static __forceinline__ void load(const float *p, float (&v)[8]) {
        asm("ld.global.nc.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
            : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "l"(p));
    }
    __device__ static __forceinline__ void store(float *p, const float (&v)[8]) {
        reinterpret_cast<float4 *>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
        reinterpret_cast<float4 *>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
    }
};

template <> struct RowVec<__nv_bfloat16, 4> {
    static constexpr int kElems = 4;
    __device__ static __forceinline__ void load(const __nv_bfloat16 *p, float (&v)[4]) {
        const uint2 t = __ldg(reinterpret_cast<const uint2 *>(p));
        v[0] = __uint_as_float(t.x << 16); v[1] = __uint_as_float(t.x & 0xffff0000u);
        v[2] = __uint_as_float(t.y << 16); v[3] = __uint_as_float(t.y & 0xffff0000u);
    }
    __device__ static __forceinline__ void store(__nv_bfloat16 *p, const float (&v)[4]) {
        const __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]), b = __floats2bfloat162_rn(v[2], v[3]);
        *reinterpret_cast<uint2 *>(p) = make_uint2(*reinterpret_cast<const unsigned *>(&a),
                                                   *reinterpret_cast<const unsigned *>(&b));
    }
};

template <> struct RowVec<__nv_bfloat16, 8> {
    static constexpr int kElems = 8;
    __device__ static __forceinline__ void load(const __nv_bfloat16 *p, float (&v)[8]) {
        const uint4 t = __ldg(reinterpret_cast<const uint4 *>(p));
        const unsigned u[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {                     // bf16 -> fp32 is a 16-bit left shift
            v[2 * i] = __uint_as_float(u[i] << 16);
            v[2 * i + 1] = __uint_as_float(u[i] & 0xffff0000u);
        }
    }
    __device__ static __forceinline__ void store(__nv_bfloat16 *p, const float (&v)[8]) {
        unsigned u[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
            u[i] = *reinterpret_cast<const unsigned *>(&h);
        }
        *reinterpret_cast<uint4 *>(p) = make_uint4(u[0], u[1], u[2], u[3]);
    }
};

// Vector reduction into global memory: one 16-byte red per call (sm_90+), no return value.
__device__ __forceinline__ void red_add_v4(float *addr, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// 4 bf16 lanes of a grad_value row, added in place (8-byte packed red, round-to-nearest; sm_90+): used by the bf16
// backward for the FINE levels, whose rows collect few contributions (see msda_bwd_tiled, MIXED).
__device__ __forceinline__ void red_add_bf16x4(__nv_bfloat16 *addr, float a, float b, float c, float d) {
    const __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
    asm volatile("red.global.add.noftz.v2.bf16x2 [%0], {%1, %2};" ::"l"(addr), "r"(*reinterpret_cast<const unsigned *>(&lo)),
                 "r"(*reinterpret_cast<const unsigned *>(&hi)) : "memory");
}

// One corner of the MIXED bf16 backward without control flow: exactly one of the two reds executes (or none when the
// corner weight is zero).  Straight-line predicated code keeps the four row loads of a tap ahead of the reds; an
// if / else around two different red instructions made ptxas serialise load -> branch -> red per corner (+45 % run time).
__device__ __forceinline__ void red_add_mixed(bool to_bf16, __nv_bfloat16 *a16, bool to_f32, float *a32, float a, float b,
                                              float c, float d) {
    const __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
    asm volatile(
        "{\n\t.reg .pred p16, p32;\n\t"
        "setp.ne.b32 p16, %0, 0;\n\t"
        "setp.ne.b32 p32, %1, 0;\n\t"
        "@p16 red.global.add.noftz.v2.bf16x2 [%2], {%3, %4};\n\t"
        "@p32 red.global.add.v4.f32 [%5], {%6, %7, %8, %9};\n\t}"
        ::"r"((unsigned)to_bf16), "r"((unsigned)to_f32), "l"(a16), "r"(*reinterpret_cast<const unsigned *>(&lo)),
          "r"(*reinterpret_cast<const unsigned *>(&hi)), "l"(a32), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

}  // namespace msda
