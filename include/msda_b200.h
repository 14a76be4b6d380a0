/*
 * msda_b200.h -- C ABI of the B200-native multi-scale deformable attention library (libmsda_b200.so).
 *
 * This is the drop-in boundary for the reference's native module `MultiScaleDeformableAttention`
 * (projects/UNINEXT/uninext/models/deformable_detr/ops/src/vision.cpp:13-16), whose two functions
 *     ms_deform_attn_forward  (ops/src/ms_deform_attn.h:19-39  -> ops/src/cuda/ms_deform_attn_cuda.cu:20-80)
 *     ms_deform_attn_backward (ops/src/ms_deform_attn.h:41-62  -> ops/src/cuda/ms_deform_attn_cuda.cu:83-153)
 * take ATen tensors. Here the same work is exposed with plain pointers and sizes; no torch / ATen type crosses
 * this interface. The reference-side binding (a 40-line pybind or ctypes shim) is shown in INTEGRATION.md and
 * shipped as uninext_b200/dropin/MultiScaleDeformableAttention.py.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer on the current CUDA device, dense row-major.  16-byte aligned tensors (what
 *     any allocator returns) take the tiled / slab sm_100a kernels; a merely element-aligned pointer (a contiguous view
 *     with a storage offset, which the reference accepts too) is served by the generic kernels:
 *       value              [N, S, M, D]          (reference: ms_deform_attn_cuda.cu:40-43)
 *       spatial_shapes     [L, 2] int64 (H_l,W_l)  -- read on the device, no host sync (cu:67)
 *       level_start_index  [L]    int64            (cu:68)
 *       sampling_loc       [N, Lq, M, L, P, 2]   last dim (x, y) in [0,1] of the level map (cu:69)
 *       attn_weight        [N, Lq, M, L, P]      (cu:70)
 *       out / grad_out     [N, Lq, M*D]          (cu:54,77)
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream). Calls are asynchronous with
 *     respect to the host, stateless and re-entrant (reference: at::cuda::getCurrentCUDAStream(), cu:65,135).
 *   - return value: 0 on success; a positive cudaError_t if a CUDA call or kernel launch failed (the reference
 *     only printf()s these, ms_deform_im2col_cuda.cuh:948-952,1321-1325 -- here they are returned);
 *     a negative MSDA_E_* for argument errors. msda_strerror() renders either.
 *   - there is no im2col_step: the reference chunks the batch only to bound its int32 indexing and temporary
 *     sizes (cu:50-52,61-75); these kernels use 64-bit offsets and take the whole batch in one launch. The
 *     Python shim still validates `batch % min(batch, im2col_step) == 0` like the reference (cu:52).
 *   - the *_bf16 entry points are new (the reference dispatches float/double only, cu:64,134): value, out and
 *     grad_out are bfloat16 bit patterns (uint16_t), sampling_loc / attn_weight and their gradients stay fp32,
 *     accumulation is fp32.
 *   - backward: grad_value is zero-filled by the callee (the reference's at::zeros_like, cu:121); grad_sampling_loc
 *     and grad_attn_weight are fully overwritten. grad_value accumulation order is not deterministic (fp32 atomics),
 *     like the reference: grad_value agrees between runs only to rounding.  grad_sampling_loc and grad_attn_weight are
 *     run-to-run stable for a given kernel selection; the forward has no atomics and is deterministic.
 *   - msda_backward_det_* are the bit-reproducible backward (what torch.use_deterministic_algorithms(True) selects in
 *     the Python shim): grad_value is accumulated as 64-bit fixed point, so it is bit-identical across runs, kernel
 *     selections (tiled / generic, SPLIT, TMA, knobs) and GPUs.  See DESIGN.md section 11.
 */
#ifndef MSDA_B200_H_
#define MSDA_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSDA_ABI_VERSION 3   /* 2: round-2 entry points (knobs, CondInst head, geometry, W-stationary GEMM); 3: deterministic backward */

#define MSDA_E_BADARG   (-1)   /* null pointer, non-positive dimension, unknown knob                  */
#define MSDA_E_TOOLARGE (-2)   /* a dimension product exceeds what the kernels index (see msda_b200.h) */
#define MSDA_E_NODEVICE (-3)   /* no sm_100 device is current                                          */

int msda_abi_version(void);
const char *msda_strerror(int code);

/* Which kernel family a (dtype, D, L, P) problem is routed to: 1 = tiled sm_100a fast path, 0 = generic.
 * dtype_bytes: 2 (bf16), 4 (fp32), 8 (fp64). Used by the tests to prove the fast path is the one exercised. */
int msda_uses_fast_path(int dtype_bytes, int D, int L, int P);

/* Number of kernel launches (memsets excluded) this process has issued through this library. */
uint64_t msda_launch_count(void);

/* Kernel-selection knobs (process-wide; initial values come from the environment variables of the same name with an
 * MSDA_ prefix, e.g. MSDA_SLAB=0).  They never change results, only which kernel computes them; the tests use
 * them to run every kernel family on small shapes, the tools to sweep them.  Returns the previous value, or
 * MSDA_E_BADARG for an unknown knob.  value == MSDA_KNOB_QUERY reads without writing.
 *   MSDA_KNOB_SLAB          1 = slab-ordered kernels (msda_slab.cuh) whenever D == 32 and L*P <= 16; 2 = tiled forward +
 *                           backward with tensor-memory accumulators for the coarse levels (msda_tmem.cuh); -1 (auto) and
 *                           0 = tiled kernels
 *   MSDA_KNOB_BWD_WIN_ROWS  shared-memory window of the slab backward in rows of 128 B (-1 = all that fits)
 *   MSDA_KNOB_BWD_LIST_CAP  entries per row-class list of the slab backward (even, >= 8)
 *   MSDA_KNOB_FWD_SLAB_CTAS resident CTAs per SM of the slab forward (1 or 2)
 *   MSDA_KNOB_F32_VEC8_FWD / _BWD   lane shape of the fp32 tiled kernels: 1 = 4 lanes x 32 B per row, 0 = 8 lanes x 16 B
 *   MSDA_KNOB_BF16_FINE_ROWS        msda_backward_bf16 with a bf16 result: levels of at least this many rows accumulate
 *                                   grad_value directly in bf16 (packed 8-byte reds); the others in fp32.  0 = all fp32.
 *                                   (changes results within the 1e-2 bf16 tolerance, see DESIGN.md.)
 *   MSDA_KNOB_BF16_PACKED_FWD       bf16 forward (D = 32 / 64, large launches): blend the 4 corners of a tap in packed bf16 and
 *                                   accumulate taps in fp32 (~3 extra bf16 roundings per tap; also changes results slightly).
 *   MSDA_KNOB_ZERO_FILL             how msda_backward_* zero-fills grad_value (results identical): 0 = cudaMemsetAsync,
 *                                   1 = msda_zero_fill kernel (16-byte stores, one wave), 2 = the same kernel launched as the
 *                                   programmatic-dependent-launch primary of the tiled backward kernel, whose prologue then
 *                                   overlaps the fill (not while the stream is being captured into a CUDA graph).  Default 2
 *                                   (cfg2 on B200: step 4.186 -> 4.156 ms, decoder-shaped backward 26.7 -> 23.6 us). */
#define MSDA_KNOB_SLAB          0
#define MSDA_KNOB_BWD_WIN_ROWS  1
#define MSDA_KNOB_BWD_LIST_CAP  2
#define MSDA_KNOB_FWD_SLAB_CTAS 3
#define MSDA_KNOB_F32_VEC8_FWD  4   /* fp32 tiled forward: 8 channels per lane (LDG.256), D in {32, 64}; 0 / 1        */
#define MSDA_KNOB_F32_VEC8_BWD  5   /* fp32 tiled backward: same lane shape; 0 / 1                                     */
#define MSDA_KNOB_BF16_FINE_ROWS 6  /* bf16 backward: levels with H*W >= this accumulate grad_value in bf16; 0 = off */
#define MSDA_KNOB_BF16_PACKED_FWD 7 /* bf16 forward: corners of a tap blended in packed bf16 (HFMA2); 0 / 1            */
#define MSDA_KNOB_ZERO_FILL     8   /* grad_value zero-fill of the backward: 0 cudaMemsetAsync, 1 own kernel, 2 own kernel
                                       as the PDL primary of the tiled backward kernel (prologue overlaps the fill)   */
#define MSDA_KNOB_COUNT         9
#define MSDA_KNOB_QUERY         (-1000000)
int msda_set_knob(int knob, int value);

/* ---- forward: replaces ms_deform_attn_cuda_forward (ms_deform_attn_cuda.cu:20-80) ---- */
int msda_forward_f32(const float *value, const int64_t *spatial_shapes, const int64_t *level_start_index,
                     const float *sampling_loc, const float *attn_weight,
                     int N, int S, int M, int D, int L, int Lq, int P,
                     float *out, void *stream);
int msda_forward_f64(const double *value, const int64_t *spatial_shapes, const int64_t *level_start_index,
                     const double *sampling_loc, const double *attn_weight,
                     int N, int S, int M, int D, int L, int Lq, int P,
                     double *out, void *stream);
int msda_forward_bf16(const uint16_t *value, const int64_t *spatial_shapes, const int64_t *level_start_index,
                      const float *sampling_loc, const float *attn_weight,
                      int N, int S, int M, int D, int L, int Lq, int P,
                      uint16_t *out, void *stream);

/* ---- backward: replaces ms_deform_attn_cuda_backward (ms_deform_attn_cuda.cu:83-153) ---- */
int msda_backward_f32(const float *grad_out, const float *value,
                      const int64_t *spatial_shapes, const int64_t *level_start_index,
                      const float *sampling_loc, const float *attn_weight,
                      int N, int S, int M, int D, int L, int Lq, int P,
                      float *grad_value, float *grad_sampling_loc, float *grad_attn_weight, void *stream);
int msda_backward_f64(const double *grad_out, const double *value,
                      const int64_t *spatial_shapes, const int64_t *level_start_index,
                      const double *sampling_loc, const double *attn_weight,
                      int N, int S, int M, int D, int L, int Lq, int P,
                      double *grad_value, double *grad_sampling_loc, double *grad_attn_weight, void *stream);
/* bf16 backward accumulates grad_value in fp32: `grad_value_f32` [N,S,M,D] fp32 is the accumulator (zero-filled by
 * the callee) and `grad_value` receives its bf16 rounding. Pass grad_value == NULL to keep only the fp32 result.
 * With MSDA_KNOB_BF16_FINE_ROWS > 0 and grad_value != NULL the big ("fine") levels are accumulated directly in
 * `grad_value` and only the rows of the coarse levels of `grad_value_f32` are used (as scratch). */
int msda_backward_bf16(const uint16_t *grad_out, const uint16_t *value,
                       const int64_t *spatial_shapes, const int64_t *level_start_index,
                       const float *sampling_loc, const float *attn_weight,
                       int N, int S, int M, int D, int L, int Lq, int P,
                       float *grad_value_f32, uint16_t *grad_value,
                       float *grad_sampling_loc, float *grad_attn_weight, void *stream);

/* ---- deterministic backward: same arguments and results as msda_backward_f32 / _bf16, bit-reproducible grad_value ----
 * `acc` is caller-allocated int64 scratch of MSDA_DET_HEADER_WORDS + N*S*M*D words, 8-byte aligned (zero-filled by the
 * callee); its header holds max|attn_weight|, max|grad_out| and a non-finite flag, the rest the fixed-point sums.  grad_value
 * (fp32) / grad_value_f32 (bf16) must not alias it.  For bf16, grad_value_f32 is scratch for non-finite contributions and
 * receives the fp32 result only when grad_value == NULL.  No host synchronisation: capture-safe.
 * Every contribution fp32(fp32(corner_weight * attn) * grad_out) is rounded to the nearest multiple of a power-of-two quantum
 * 2^(e + ceil(log2(Lq*L*P)) - 62), with 2^e >= max|attn| * max|grad_out|, and summed exactly; NaN / +-Inf contributions are
 * summed in IEEE fp32 apart (order-independent) and added at the end.  The kernel-selection knobs SLAB, F32_VEC8_BWD and
 * BF16_FINE_ROWS do not apply here; the tiled kernels (linear / TMA / SPLIT) and the generic kernel are chosen as in the
 * default path and give identical bits.  There is no deterministic fp64 backward. */
#define MSDA_DET_HEADER_WORDS 4
int msda_backward_det_f32(const float *grad_out, const float *value,
                          const int64_t *spatial_shapes, const int64_t *level_start_index,
                          const float *sampling_loc, const float *attn_weight,
                          int N, int S, int M, int D, int L, int Lq, int P,
                          int64_t *acc, float *grad_value, float *grad_sampling_loc, float *grad_attn_weight, void *stream);
int msda_backward_det_bf16(const uint16_t *grad_out, const uint16_t *value,
                           const int64_t *spatial_shapes, const int64_t *level_start_index,
                           const float *sampling_loc, const float *attn_weight,
                           int N, int S, int M, int D, int L, int Lq, int P,
                           int64_t *acc, float *grad_value_f32, uint16_t *grad_value,
                           float *grad_sampling_loc, float *grad_attn_weight, void *stream);

/* ---- callers of the op (SURVEY.md section 8 rows f-1 / f-2): one-pass fp32 kernels around the cuBLAS GEMMs --------
 * msda_prologue_forward_f32: raw projection -> attention softmax + sampling locations in the op's layouts.
 *   Replaces the five elementwise passes of ops/modules/ms_deform_attn.py:99-112.
 *   proj [R, M*L*P*3]: columns [0, M*L*P*2) = sampling offsets ordered (m,l,p,xy) (ms_deform_attn.py:99),
 *                      columns [M*L*P*2, M*L*P*3) = attention logits ordered (m, l*p) (ms_deform_attn.py:100);
 *   ref  [R, L, refdim] reference points (refdim 2) or boxes (refdim 4) (ms_deform_attn.py:103-109); R = N*Lq;
 *   loc  [R, M, L, P, 2], attn [R, M, L, P] outputs.  L*P <= 32.
 * msda_prologue_backward_f32: gradient of the raw projection from grad_loc / grad_attn (reference points are
 *   treated as constants).
 * msda_colsum_f32: out[c] = sum_r x[r,c] (bias gradients); cols % 4 == 0; `out` is zero-filled by the callee.
 * msda_add_layernorm_forward_f32 / msda_layernorm_backward_f32: y = LayerNorm(a + b) over the last dimension
 *   (deformable_transformer.py:354-356,359); cols in {128, 256, 384, 512}; b and z may be NULL (z = a + b is needed by
 *   the backward when b != NULL); dgamma / dbeta are zero-filled by the callee. */
int msda_prologue_forward_f32(const float *proj, const float *ref, const int64_t *spatial_shapes,
                              int64_t R, int M, int L, int P, int refdim, float *loc, float *attn, void *stream);
int msda_prologue_backward_f32(const float *grad_loc, const float *grad_attn, const float *attn, const float *ref,
                               const int64_t *spatial_shapes, int64_t R, int M, int L, int P, int refdim,
                               float *grad_proj, void *stream);
int msda_colsum_f32(const float *x, int64_t rows, int cols, float *out, void *stream);
/* ReLU backward fused with the bias gradient of the Linear before it (FFN linear1): g2 = g where y > 0 else 0;
 * colsum[c] = sum_r g2[r, c] (zero-filled by the callee).  cols % 4 == 0. */
int msda_relu_backward_colsum_f32(const float *g, const float *y, int64_t rows, int cols, float *g2, float *colsum, void *stream);
/* Deterministic variants (no float atomics; what torch.use_deterministic_algorithms(True) selects in the Python wrappers):
 * each CTA writes its partial row, summed in a fixed order, to caller-allocated `scratch`, and a second kernel adds the rows
 * in index order.  The grid depends only on (rows, cols), so results are bit-identical across runs and GPUs.  Scratch
 * sizes come from the host-only query functions (0 and *bytes on success, MSDA_E_BADARG on bad arguments); scratch must be
 * 16-byte aligned.  The results are fully written (no zero-fill needed). */
int msda_colsum_det_scratch_bytes(int64_t rows, int cols, int64_t *bytes);    /* colsum and relu_backward_colsum */
int msda_layernorm_backward_det_scratch_bytes(int64_t rows, int cols, int64_t *bytes);
int msda_colsum_det_f32(const float *x, int64_t rows, int cols, float *scratch, float *out, void *stream);
int msda_relu_backward_colsum_det_f32(const float *g, const float *y, int64_t rows, int cols, float *g2, float *scratch,
                                      float *colsum, void *stream);
int msda_layernorm_backward_det_f32(const float *dy, const float *z, const float *gamma, const float *mean,
                                    const float *rstd, int64_t rows, int cols, float *dz, float *scratch, float *dgamma,
                                    float *dbeta, void *stream);
int msda_add_layernorm_forward_f32(const float *a, const float *b, const float *gamma, const float *beta,
                                   int64_t rows, int cols, float eps, float *z, float *y, float *mean, float *rstd,
                                   void *stream);
int msda_layernorm_backward_f32(const float *dy, const float *z, const float *gamma, const float *mean,
                                const float *rstd, int64_t rows, int cols, float *dz, float *dgamma, float *dbeta,
                                void *stream);

/* ---- geometry feeding the op (SURVEY.md section 8 f-3; deformable_transformer_dino.py:132-171,289-301,612-646): one launch each
 *   msda_valid_counts:            mask [N, S] bytes (non-zero = padded) -> counts [N, L, 2] int32 = (valid_W, valid_H)  (get_valid_ratio)
 *   msda_encoder_ref_points_f32:  valid_ratios [N, L, 2] -> reference points [N, S, L, 2]                          (get_reference_points)
 *   msda_encoder_proposals_f32:   mask + counts -> proposals [N, S, 4] in logit space (+inf = dropped), keep [N, S] bytes
 *                                 (the geometry half of gen_encoder_output_proposals)
 *   msda_sine_pos_embed_forward/backward_f32: pos [R, n] -> [R, n * F]                                              (get_sine_pos_embed) */
int msda_valid_counts(const uint8_t *mask, const int64_t *spatial_shapes, const int64_t *level_start_index, int N, int S, int L,
                      int32_t *counts, void *stream);
int msda_encoder_ref_points_f32(const float *valid_ratios, const int64_t *spatial_shapes, const int64_t *level_start_index, int N,
                                int S, int L, float *ref, void *stream);
int msda_encoder_proposals_f32(const uint8_t *mask, const int32_t *counts, const int64_t *spatial_shapes,
                               const int64_t *level_start_index, int N, int S, int L, float base_scale, float *proposals,
                               uint8_t *keep, void *stream);
int msda_sine_pos_embed_forward_f32(const float *pos, int64_t R, int n, int F, float temperature, int exchange_xy, float *out,
                                    void *stream);
int msda_sine_pos_embed_backward_f32(const float *pos, const float *grad_out, int64_t R, int n, int F, float temperature,
                                     int exchange_xy, float *grad_pos, void *stream);

/* ---- CondInst dynamic mask head (SURVEY.md section 8 f-4; uninext/models/ddetrs.py:488-598, 895-958) ----------------
 * msda_condinst_forward_f32: logits[i, y, x] = MLP_i(rel_x, rel_y, feats[b(i), :, y, x]) for every selected instance i --
 *   the reference's three grouped 1x1 convolutions (groups = #instances, `mask_heads_forward`) over a materialised
 *   [1, I*10, H, W] input, fused into one pass that materialises nothing.
 *     feats [N, 8, H, W]; params [I, 169] laid out as parse_dynamic_params expects (w1[8][10] | w2[8][8] | w3[8] | b1 | b2 | b3);
 *     refs [I, 2] reference points in input-image pixels; inst_start [N + 1] int32 (device): instances of image b are
 *     [inst_start[b], inst_start[b+1]); max_inst = largest per-image count (host value, sizes the grid);
 *     stride = mask_feat_stride; rel_coord = 1 prepends (ref - pixel location) as two input channels, 0 feeds zeros;
 *     logits [I, H, W].
 * msda_condinst_backward_f32: grad_feats [N, 8, H, W], grad_params [I, 169] and grad_refs [I, 2] (all zero-filled by the
 *   callee, then accumulated with fp32 reductions: summation order, hence the last bits, vary from run to run;
 *   msda_condinst_backward_det_f32 below is the bit-reproducible variant).
 * msda_aligned_bilinear_forward/backward_f32: `aligned_bilinear` (ddetrs.py:921-942) on [planes, h, w] -> [planes, f*h, f*w]. */
int msda_condinst_forward_f32(const float *feats, const float *params, const float *refs, const int32_t *inst_start,
                              int N, int H, int W, int I, int max_inst, int stride, int rel_coord, float *logits,
                              void *stream);
int msda_condinst_backward_f32(const float *grad_logits, const float *feats, const float *params, const float *refs,
                               const int32_t *inst_start, int N, int H, int W, int I, int max_inst, int stride,
                               int rel_coord, float *grad_feats, float *grad_params, float *grad_refs, void *stream);
/* Deterministic CondInst backward: same arguments and results as msda_condinst_backward_f32 plus caller scratch of
 * msda_condinst_backward_det_scratch_bytes() bytes (per-instance-chunk feature partials and per-warp parameter partials,
 * added in a fixed order by a second kernel); no float atomics, bit-identical across runs and GPUs. */
int msda_condinst_backward_det_scratch_bytes(int N, int H, int W, int I, int max_inst, int64_t *bytes);
int msda_condinst_backward_det_f32(const float *grad_logits, const float *feats, const float *params, const float *refs,
                                   const int32_t *inst_start, int N, int H, int W, int I, int max_inst, int stride,
                                   int rel_coord, float *scratch, float *grad_feats, float *grad_params, float *grad_refs,
                                   void *stream);
int msda_aligned_bilinear_forward_f32(const float *in, int64_t planes, int h, int w, int factor, float *out, void *stream);
int msda_aligned_bilinear_backward_f32(const float *grad_out, int64_t planes, int h, int w, int factor, float *grad_in,
                                       void *stream);

/* ---- tcgen05 GEMM for the Linears that bracket the op:  C[M,N] = A[M,K] . W[N,K]^T + bias[N]  (fp32 storage, TF32 MMA
 * with fp32 accumulation in tensor memory; TMA-fed).  K % 32 == 0, N % 32 == 0 (N % 64 == 0 above 256), N <= 512.
 * Replaces torch.nn.functional.linear for value_proj / output_proj / the concatenated sampling projection
 * (ops/modules/ms_deform_attn.py:95,99-100,115) when TF32 GEMMs are allowed. bias may be NULL. */
int msda_linear_tf32(const float *A, const float *W, const float *bias, int64_t M, int N, int K, float *C, void *stream);
/* W-stationary variant with a fused tail, for K <= 256 and N <= 256 (N % 64 == 0; msda_linear_tf32_ws_ok tells):
 *   C = A . W^T + bias;  rows with row_mask[m] != 0 are written as zeros (the `masked_fill(input_padding_mask)` that follows
 *   value_proj, ops/modules/ms_deform_attn.py:96-97);  relu != 0 applies max(., 0) (FFN linear1).  bias / row_mask may be NULL.
 *   msda_linear_tf32 itself routes eligible shapes to this kernel.  Two implementations: for K <= 256 a 2-CTA MMA kernel
 *   (tcgen05.mma.cta_group::2, M = 256 per CTA pair, TMA-store epilogue), otherwise / with MSDA_GEMM_WS2=0 the 1-CTA kernel
 *   with multicast A.  A, W, C (and bias) must be 16-byte aligned. */
int msda_linear_tf32_ex(const float *A, const float *W, const float *bias, const uint8_t *row_mask, int64_t M, int N, int K,
                        int relu, float *C, void *stream);
int msda_linear_tf32_ws_ok(int N, int K);
/* Diagnostic: phase timeline of the last 2-CTA W-stationary GEMM launched with MSDA_GEMM_WS_DBG=1 (160 CTAs x 24 slots of
 * SM-clock stamps; layout in msda_gemm_sm100.cu).  Copies min(n_words, 3840) words to `out` (host). */
int msda_debug_gemm_timeline(unsigned long long *out, int n_words);

#ifdef __cplusplus
}
#endif
#endif /* MSDA_B200_H_ */
