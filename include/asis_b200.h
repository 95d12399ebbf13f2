/* asis_b200.h -- C ABI of libasis_b200.so: the B200 (sm_100a) kernels behind the AdapterSIS
 * encoder hot path.
 *
 * The reference (weimengmeng1999/AdapterSIS) has no native boundary at all: its deformable
 * attention "op" is a Python loop over F.grid_sample (backbones/ops/modules/ms_deform_attn.py:33-54)
 * and every dense op is an nn.Module calling ATen.  The historical native boundary of this op
 * family is MSDeformAttnFunction.apply (ms_deform_attn.py:17-30, call site :176-183); this header
 * is what a replacement for that boundary -- and for the dense ops next to it -- exports.
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless named *_host;
 *   - the caller owns every buffer, including workspaces (sized by the matching
 *     *_workspace_bytes function); nothing here allocates or frees device memory;
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*); no entry point
 *     synchronises; the library is re-entrant across streams;
 *   - return value 0 = enqueued; negative = ASIS_ERR_*; asis_last_error() returns a
 *     thread-local, human-readable message for the last failure on the calling thread;
 *   - dtype arguments: ASIS_F32 = 0, ASIS_BF16 = 1.  "compute mode" ASIS_F32 uses fp32 FFMA
 *     kernels (parity mode, 1e-4), ASIS_BF16 uses tcgen05 tensor-core kernels with bf16
 *     operands and fp32 accumulation (performance mode, 2e-2).
 */
#ifndef ASIS_B200_H_
#define ASIS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ASIS_ABI_VERSION 1

enum { ASIS_F32 = 0, ASIS_BF16 = 1 };

enum {
  ASIS_OK = 0,
  ASIS_ERR_INVALID = -1,   /* bad argument (shape, dtype, alignment, null pointer) */
  ASIS_ERR_WORKSPACE = -2, /* workspace too small */
  ASIS_ERR_CUDA = -3,      /* a CUDA runtime / driver call failed */
  ASIS_ERR_UNSUPPORTED = -4
};

/* Operand majors for asis_gemm (which dimension is contiguous in memory). */
enum { ASIS_MAJOR_K = 0, ASIS_MAJOR_MN = 1 };

/* Epilogues for asis_gemm.  acc = sum_k A[m,k]*B[n,k] (fp32). */
enum {
  ASIS_EPI_NONE = 0,          /* C = acc (+ bias)                                             */
  ASIS_EPI_GELU = 1,          /* aux = acc + bias (pre-activation, optional); C = gelu_erf(aux) */
  ASIS_EPI_SCALE_RESIDUAL = 2,/* aux = acc + bias (optional); C = residual + gamma[n] * aux     */
  ASIS_EPI_DGELU = 3,         /* C = acc * gelu_erf'(aux_in)      (aux is an INPUT here)        */
  ASIS_EPI_ACCUMULATE = 4,    /* C += acc   (fp32 C only; weight-gradient accumulation)       */
  ASIS_EPI_GELU_GRAD = 5,     /* h = acc + bias; C = gelu_erf(h); aux = gelu_erf'(h)  (aux required): the forward
                                 saves the derivative -- it shares the erfc / exp evaluation with the activation --
                                 so that the backward epilogue below is a multiply                               */
  ASIS_EPI_MUL_AUX = 6        /* C = acc * aux_in   (aux is an INPUT: the derivative saved by GELU_GRAD)          */
};

int asis_abi_version(void);
const char *asis_last_error(void);
/* Number of kernels this library has launched on the calling process since load (bench.py's
 * gpu_launches claim is read from here). */
uint64_t asis_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Multi-scale deformable attention  --  replaces ms_deform_attn_core_pytorch
 * (ms_deform_attn.py:33-54) behind MSDeformAttnFunction.apply (:17-30).
 *
 *   value            [N, S, M, D]          value_dtype (f32 | bf16)
 *   spatial_shapes   [L, 2] int64 (H, W)   device memory, as the reference passes it
 *   level_start      [L]    int64          device memory (the reference ignores it, :26; here it
 *                                          is used, so it must be the exclusive cumsum of H*W)
 *   sampling_loc     [N, Lq, M, L, P, 2]   f32, (x, y) normalised to [0,1]
 *   attn_weight      [N, Lq, M, L, P]      f32
 *   out              [N, Lq, M*D]          out_dtype
 * Pixel coordinate = loc * size - 0.5, bilinear, zero padding (grid_sample align_corners=False).
 * D must be a multiple of 4 (f32) / 8 (bf16); L <= 8; L*P <= 64.
 * ------------------------------------------------------------------------------------------ */
int asis_msda_forward(const void *value, int value_dtype, const int64_t *spatial_shapes,
                      const int64_t *level_start, const float *sampling_loc,
                      const float *attn_weight, void *out, int out_dtype, int N, int S, int M,
                      int D, int Lq, int L, int P, void *stream);

/* Backward (the reference's Function has none, SURVEY.md F2; semantics = autograd through the
 * reference core).  No floating-point atomics, run-to-run deterministic: the contributions to
 * grad_value are indexed per value pixel (integer count -> scan -> ordered fill), then one thread
 * group per pixel sums its list in a fixed order and writes each element exactly once.
 *   grad_out     [N, Lq, M*D]  gdtype      grad_value  [N, S, M, D]  gdtype (fully overwritten)
 *   grad_loc     [N, Lq, M, L, P, 2] f32   grad_attn   [N, Lq, M, L, P] f32
 */
size_t asis_msda_backward_workspace_bytes(int N, int S, int M, int D, int Lq, int L, int P);
int asis_msda_backward(const void *value, int value_dtype, const int64_t *spatial_shapes,
                       const int64_t *level_start, const float *sampling_loc,
                       const float *attn_weight, const void *grad_out, int gdtype,
                       void *grad_value, float *grad_loc, float *grad_attn, int N, int S, int M,
                       int D, int Lq, int L, int P, void *workspace, size_t workspace_bytes,
                       void *stream);

/* Fused softmax(L*P) + sampling-location arithmetic of MSDeformAttn.forward (:156-171):
 *   logits [R, M*L*P] -> attn [R, M, L, P] = softmax over L*P;
 *   offsets [R, M, L, P, 2] + reference points -> loc = ref + off / (W_l, H_l)     (ref_dim 2)
 *                                                 loc = ref.xy + off / P * ref.wh * 0.5 (ref_dim 4)
 *   ref [Rr, Lr, ref_dim] with Rr in {R, Lq} (broadcast over batch) and Lr in {L, 1}.
 * and its backward (grad_loc, grad_attn -> grad_offsets, grad_logits). */
int asis_msda_prep_forward(const void *offsets, const void *logits, int in_dtype, const float *ref,
                           int ref_rows, int ref_levels, int ref_dim, const int64_t *spatial_shapes,
                           float *loc, float *attn, int R, int Lq, int M, int L, int P, void *stream);
int asis_msda_prep_backward(const float *grad_loc, const float *grad_attn, const float *attn,
                            const float *ref, int ref_rows, int ref_levels, int ref_dim,
                            const int64_t *spatial_shapes, void *grad_offsets, void *grad_logits,
                            int out_dtype, int R, int Lq, int M, int L, int P, void *stream);

/* ------------------------------------------------------------------------------------------
 * LayerNorm (nn.LayerNorm(eps=1e-6): dinov2/models/vision_transformer.py:89,
 * backbones/adapter_blocks.py:114,118-119,127,163-164).
 *   x [R, C] x_dtype -> y [R, C] y_dtype; mean/rstd [R] f32 saved for backward.
 * Backward: dx = (dres ? dres : 0) + LN'(dy); partial dgamma/dbeta in workspace, reduced in
 * fixed order (deterministic) into dgamma/dbeta (accumulate != 0 adds to existing contents).
 * ------------------------------------------------------------------------------------------ */
int asis_layernorm_forward(const void *x, int x_dtype, const float *gamma, const float *beta,
                           void *y, int y_dtype, float *mean, float *rstd, int R, int C, float eps,
                           void *stream);
size_t asis_layernorm_backward_workspace_bytes(int R, int C);
int asis_layernorm_backward(const void *dy, int dy_dtype, const void *x, int x_dtype,
                            const float *gamma, const float *mean, const float *rstd,
                            const float *dres, float *dx, float *dgamma, float *dbeta,
                            int accumulate, int R, int C, void *workspace, size_t workspace_bytes,
                            void *stream);

/* ------------------------------------------------------------------------------------------
 * Dense contraction  C[M,N] = epilogue( sum_k A[m,k] * B[n,k] )        (nn.Linear and its grads)
 *   compute ASIS_BF16: A, B bf16; tcgen05.mma (kind::f16) with TMA-fed 128B-swizzled tiles,
 *                      fp32 accumulators in TMEM.  lda/ldb/ldc in elements; pointers 16-byte
 *                      aligned, leading dimensions multiples of 8.
 *   compute ASIS_F32 : A, B f32; FFMA tiles (parity mode).
 *   a_major/b_major: ASIS_MAJOR_K  -> operand stored [rows, K] (K contiguous, ld = row pitch)
 *                    ASIS_MAJOR_MN -> operand stored [K, rows] (rows contiguous, ld = k pitch)
 *   bias [N] f32 (nullable), gamma [N] f32, residual [M, ldc] f32, aux [M, ldaux] aux_dtype.
 *   Forward Linear: A=x(K-major), B=W[out,in](K-major).  dgrad: A=dy(K), B=W(MN).
 *   wgrad: A=dy(MN), B=x(MN), epilogue ACCUMULATE.
 * ------------------------------------------------------------------------------------------ */
int asis_gemm(int compute, const void *A, int a_major, int64_t lda, const void *B, int b_major,
              int64_t ldb, void *C, int c_dtype, int64_t ldc, int M, int N, int K, int epilogue,
              const float *bias, const float *gamma, const float *residual, void *aux,
              int aux_dtype, int64_t ldaux, void *stream);

/* Column sums (bias gradients): out[n] (+)= sum_m X[m, n];  optionally of X*Y elementwise
 * (LayerScale gamma gradient, dinov2/layers/layer_scale.py:26-27).  Deterministic two-stage. */
size_t asis_colsum_workspace_bytes(int M, int N);
int asis_colsum(const void *X, int x_dtype, const void *Y, int y_dtype, int64_t ld, float *out,
                int accumulate, int M, int N, void *workspace, size_t workspace_bytes,
                void *stream);

/* Elementwise helpers: out = a * gamma[n] (LayerScale backward, cast), out = a + b, casts. */
int asis_scale_cols(const void *a, int a_dtype, const float *gamma, void *out, int out_dtype,
                    int64_t M, int N, void *stream);
int asis_add(const void *a, int a_dtype, const void *b, int b_dtype, void *out, int out_dtype,
             int64_t n, void *stream);
int asis_cast(const void *a, int a_dtype, void *out, int out_dtype, int64_t n, void *stream);

/* ------------------------------------------------------------------------------------------
 * Self-attention over packed qkv  (dinov2/layers/attention.py:56-69 / :73-89)
 *   qkv [B, T, 3, H, hd] -> out [B, T, H*hd];  softmax((q*hd^-0.5) k^T) v, no mask, no dropout.
 *   lse [B, H, T] f32 saved for backward.
 *   compute ASIS_BF16: flash-style tcgen05 kernel, hd == 64.
 *   compute ASIS_F32 : FFMA kernel, any hd <= 128 (parity mode).
 * Backward: dqkv [B, T, 3, H, hd] fully overwritten.
 * ------------------------------------------------------------------------------------------ */
size_t asis_attention_forward_workspace_bytes(int compute, int B, int T, int H, int hd);
int asis_attention_forward(int compute, const void *qkv, void *out, float *lse, int B, int T,
                           int H, int hd, void *workspace, size_t workspace_bytes, void *stream);
size_t asis_attention_backward_workspace_bytes(int compute, int B, int T, int H, int hd);
int asis_attention_backward(int compute, const void *qkv, const void *out, const float *lse,
                            const void *dout, void *dqkv, int B, int T, int H, int hd,
                            void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * Patch embedding front end (dinov2/layers/patch_embed.py:65-81): gather p x p patches of an
 * NCHW f32 image into rows [B*gh*gw, ldk] (k = c*p*p + dy*p + dx, zero padded to ldk) so that
 * the stride-p convolution becomes asis_gemm; and its transpose for the input gradient.
 * ------------------------------------------------------------------------------------------ */
int asis_patchify(const float *img, void *cols, int out_dtype, int B, int Cin, int Himg, int Wimg,
                  int patch, int64_t ldk, void *stream);

/* Depth-wise 3x3 convolution over token-major pyramids (backbones/adapter_blocks.py:62-80):
 *   x [B, n_tok, C] holding `n_maps` maps back to back (map i is hs[i] x ws[i]); stride 1, pad 1,
 *   weight [C, 3, 3] f32, bias [C] f32; optional fused exact GELU on the output.
 *   hs_host/ws_host are HOST arrays.  C % 4 == 0 and C <= 1280 (the forward stages the nine taps of all
 *   channels in 36 C bytes of shared memory); 1..4 maps.  x, y, pre, bias (forward) and dy, pre, x, dx,
 *   workspace (backward) must be 16-byte aligned. */
int asis_dwconv3x3_forward(const void *x, int dtype, const float *weight, const float *bias,
                           void *pre, void *y, int B, int C, int n_maps, const int *hs_host,
                           const int *ws_host, int fuse_gelu, void *stream);
size_t asis_dwconv3x3_backward_workspace_bytes(int B, int C, int n_tok);
int asis_dwconv3x3_backward(const void *dy, const void *pre, const void *x, int dtype,
                            const float *weight, void *dx, float *dweight, float *dbias,
                            int accumulate, int B, int C, int n_maps, const int *hs_host,
                            const int *ws_host, int fuse_gelu, void *workspace,
                            size_t workspace_bytes, void *stream);

/* Bilinear 2x upsampling with align_corners=True on channels-last tensors: the nn.Upsample layers of
 * FeatureDecoder (backbones/decoders.py:104-127; SURVEY.md 8f rank 2, the step after the hot path).
 *   x [B, H, W, C] -> y [B, 2H, 2W, C];  backward: gy [B, 2H, 2W, C] -> gx [B, H, W, C] (gather, no atomics).
 *   C must be a multiple of 4 (f32) / 8 (bf16). */
int asis_upsample2x_bilinear_forward(const void *x, void *y, int dtype, int B, int H, int W, int C,
                                     void *stream);
int asis_upsample2x_bilinear_backward(const void *gy, void *gx, int dtype, int B, int H, int W, int C,
                                      void *stream);
/* the same with storage padding on either side (maps [B, H + 2p, W + 2p, C], zero border): pad_in belongs to x / gx,
 * pad_out to y / gy -- the decoder keeps the maps that feed asis_conv3x3s1_gemm zero-padded */
int asis_upsample2x_bilinear_forward_padded(const void *x, void *y, int dtype, int B, int H, int W, int C,
                                            int pad_in, int pad_out, void *stream);
int asis_upsample2x_bilinear_backward_padded(const void *gy, void *gx, int dtype, int B, int H, int W,
                                             int C, int pad_in, int pad_out, void *stream);

/* The optimizer update of the step (train.py:178-189: torch.optim.SGD(momentum, weight_decay), dampening 0, no Nesterov)
 * over a list of f32 tensors:  g' = g + wd p;  buf = momentum buf + g';  p -= lr buf.   params / grads / bufs: HOST arrays
 * of n_tensors device pointers, numels their element counts; the pointer tables ride in the kernel parameters (48
 * tensors per launch), so the launches capture into a CUDA graph unchanged.  A zero-initialised buf reproduces
 * PyTorch's first step (buf = g'). */
int asis_sgd_step(int n_tensors, void *const *params, const void *const *grads, void *const *bufs,
                  const int64_t *numels, float lr, float momentum, float weight_decay, void *stream);

/* Input ingest (tools/dataset.py:111-118: np.uint8 HWC image -> torch.from_numpy(img.transpose(2, 0, 1)) / 255.0, mask
 * -> .long()) on the device: frames [B, H, W, 3] u8 -> img [B, 3, H, W] f32 = frames / 255 (IEEE division: bit-identical
 * to the host pipeline), masks [B, H, W] u8 -> target [B, H, W] i64 (both or neither).  A quarter of the host-to-device
 * bytes of the float batch. */
int asis_frames_to_batch(const uint8_t *frames, float *img, const uint8_t *masks, int64_t *target, int B, int H,
                         int W, void *stream);

/* LayerScale backward (dinov2/layers/layer_scale.py:26-27 behind x + ls(branch(x)), block.py:112-113) in
 * one pass over the incoming gradient d [M, N] f32:  du = d * gamma (dtype, the branch-output gradient),
 * dgamma = colsum(d * u) (optional, needs the saved branch output u), dbias = colsum(du) (optional: the
 * bias gradient of the branch's last nn.Linear). */
size_t asis_layerscale_backward_workspace_bytes(int M, int N);
int asis_layerscale_backward(const float *d, const void *u, const float *gamma, void *du, int dtype,
                             float *dgamma, float *dbias, int M, int N, void *workspace,
                             size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Convolutional stages either side of the hot path (SURVEY.md 8f rank 1 / 2), channels-last:
 * the spatial prior module  FeatureEncoder  (backbones/encoders.py:4-74) and  FeatureDecoder
 * (backbones/decoders.py:92-164).  A map is stored as [B, H + 2*sp, W + 2*sp, C] ("storage padding"
 * sp >= 0, zeros in the border; sp = 0 is the plain layout).  A convolution is asis_im2col + asis_gemm:
 * rows = output pixels (b, oy, ox), K = (ky, kx, c) with c fastest, weight viewed as [Cout, ky, kx, Cin];
 * its input gradient is the transposed GEMM + asis_col2im (a gather over the taps that touch an input
 * pixel: no atomics), its weight gradient the MN-major GEMM over the same column matrix.
 * ------------------------------------------------------------------------------------------ */
int asis_im2col(const void *x, int x_dtype, void *cols, int cols_dtype, int B, int H, int W, int C,
                int storage_pad, int k, int stride, int pad, int64_t ldk, void *stream);
int asis_col2im(const void *dcols, void *dx, int dtype, int B, int H, int W, int C, int storage_pad,
                int k, int stride, int pad, int64_t ldk, void *stream);

/* The 3x3 / stride 1 / pad 1 convolutions (two of the stem, the four of the decoder) as IMPLICIT GEMMs on the tcgen05
 * kernel: maps are stored zero-padded, [B, H+2, W+2, C] bf16 (storage padding 1), and tap (ky, kx) of the K loop
 * reads the A rows shifted by (ky-1)(W+2) + (kx-1) through the TMA coordinates -- no column matrix in memory.
 *   op 0: y_p [B,H+2,W+2,Cout] (c_dtype) = conv(x_p = a, w2 = b [Cout, 9*Cin] bf16, K = (ky, kx, cin)) + bias
 *   op 1: dx_p [B,H+2,W+2,Cin] (c_dtype) from dy_p = a (ZERO border) and w2 = b
 *   op 2: dw2 [Cout, 9*Cin] f32 = c from dy_p = a (ZERO border) and x_p = b
 * The border rows of the outputs of op 0 / 1 hold values of positions outside the image: read the logical pixels only.
 * Cin, Cout multiples of 64. */
int asis_conv3x3s1_gemm(int op, const void *a, const void *b, void *c, int c_dtype, const float *bias,
                        int B, int H, int W, int Cin, int Cout, void *stream);

/* BatchNorm in training mode (nn.SyncBatchNorm encoders.py:12-40, nn.BatchNorm2d decoders.py:100-125), two
 * kernels each way.  Statistics: per-channel sums over the logical pixels, fixed-order partials (no atomics):
 *   mode 0: s1 = sum (x - shift[c]),  s2 = sum (x - shift[c])^2        (shifted: no cancellation)
 *   mode 1: s1 = sum dz,  s2 = sum dz * xhat,   dz = dy * relu'(a (x - mean) + b),  xhat = (x - mean) * rstd
 * s1, s2 are the two halves of ONE [2C] f32 buffer; the cross-rank exchange of SyncBatchNorm acts on it.
 * Apply:  mode 0: y = act(a[c] (x - mean[c]) + b[c])   (a = weight * rstd, b = bias; y may use another storage
 *                                             padding; its border is zero-filled)
 *         mode 1: dx = a[c] * (dz - c1[c] - xhat * c2[c])            (c1 = mean dz, c2 = mean dz * xhat);
 *                 dx is written in storage pad_out, dy is read in storage dy_pad                         */
size_t asis_chan_stats_workspace_bytes(int B, int H, int W, int C);
int asis_chan_stats(int mode, const void *x, const void *dy, int dtype, int B, int H, int W, int C,
                    int storage_pad, int dy_pad, const float *shift, const float *a, const float *b,
                    const float *mean, const float *rstd, int relu, float *s1, float *s2,
                    void *workspace, size_t workspace_bytes, void *stream);
int asis_bn_apply(int mode, const void *x, const void *dy, int in_dtype, void *out, int out_dtype,
                  int B, int H, int W, int C, int pad_in, int pad_out, int dy_pad, const float *a,
                  const float *b, const float *mean, const float *rstd, const float *c1, const float *c2,
                  int relu, void *stream);

/* nn.MaxPool2d(kernel_size=3, stride=2, padding=1) (encoders.py:20): idx [same shape as y] u8 = winning tap
 * (first maximum in window order, as ATen); the backward is a gather over the <= 4 windows of an input pixel. */
int asis_maxpool3x3s2_forward(const void *x, void *y, uint8_t *idx, int dtype, int B, int H, int W, int C,
                              int pad_in, int pad_out, void *stream);
int asis_maxpool3x3s2_backward(const void *gy, const uint8_t *idx, void *gx, int dtype, int B, int H,
                               int W, int C, int pad_in, int pad_out, void *stream);

/* Segmentation head: nn.Upsample(scale_factor=2, bilinear, align_corners=True) followed by the 3x3 / pad 1
 * convolution to n_classes <= 4 (decoders.py:125-129: the resize of decoder_4 + final_out), fused.  Both are linear
 * and the resize acts per channel, so the C -> n_classes contraction runs FIRST, at the low resolution, and the
 * high-resolution pass interpolates and adds the nine shifted taps: the upsampled C-channel map (694 MB at the
 * reference's sizes) and its gradient are never materialised.
 *   z [B,H,W,C] channels-last, w2 [9*CO, C] f32 with row (ky*3 + kx)*CO + co, bias [CO] f32 or null,
 *   y / gy [B,2H,2W,CO] f32;  backward: gz (z's dtype, optional), gw2 [9*CO, C] f32 (optional). */
size_t asis_seg_head_workspace_bytes(int B, int H, int W, int C, int CO);
int asis_seg_head_forward(const void *z, int dtype, const float *w2, const float *bias, float *y, int B,
                          int H, int W, int C, int CO, void *workspace, size_t workspace_bytes,
                          void *stream);
int asis_seg_head_backward(const void *z, int dtype, const float *w2, const float *gy, void *gz,
                           float *gw2, int B, int H, int W, int C, int CO, void *workspace,
                           size_t workspace_bytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* ASIS_B200_H_ */
