/*
 * vp_b200.h -- C ABI of libvp_b200.so: the B200 (sm_100a) kernels behind the SAVP training path.
 *
 * The reference (alexlee-gk/video_prediction) has no FFI: its seam is the Python model registry
 * (video_prediction/models/__init__.py:12-25) whose classes call tf.nn.* primitives.  Each entry
 * point below replaces the TensorFlow primitive(s) named in its comment (file:line in the
 * reference) and is called only by the host layer in video_prediction_b200/, which keeps the
 * reference's registry / hparams / build_graph surface.  See INTEGRATION.md.
 *
 * Conventions
 *   - all tensors fp32, device pointers, NHWC / NDHWC ("channels last"), densely packed except
 *     for the channel stride (so a kernel can write into a slice of a wider concat buffer);
 *   - the caller allocates every buffer; the library never frees or retains a pointer;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), no hidden syncs;
 *   - return value 0 on success, <0 on error; vp_last_error() gives the message (thread-local).
 */
#ifndef VP_B200_H_
#define VP_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* vp_stream_t; /* cudaStream_t */

/* NDHWC view of a channel slice of an fp32 buffer.  2-D tensors use d = 1.
 * element (n,z,y,x,ch) lives at ptr[(((n*d + z)*h + y)*w + x)*cstride + ch], ch < c.
 * ptr must be 16-byte aligned and cstride a multiple of 4. */
typedef struct vp_tensor {
  float* ptr;
  int32_t n, d, h, w;
  int32_t c;       /* channels visible through this view            */
  int32_t cstride; /* channels of the underlying buffer (>= c)      */
} vp_tensor;

/* Convolution geometry.  transposed == 0:  out[o] = sum_r in[s*o + r - pad] * W[r]
 *                        transposed == 1:  out[i] = sum_{o,r : s*o + r - pad = i} in[o] * W[r]
 * Zero padding outside the input; W[r] is the "effective tap matrix" [cin][cout]. */
typedef struct vp_conv_geom {
  int32_t kd, kh, kw;
  int32_t sd, sh, sw;
  int32_t pd, ph, pw; /* pad before */
  int32_t transposed;
} vp_conv_geom;

enum { VP_ACT_NONE = 0, VP_ACT_RELU = 1, VP_ACT_LRELU = 2, VP_ACT_SIGMOID = 3, VP_ACT_TANH = 4 };
enum { VP_WKIND_PLAIN = 0, VP_WKIND_POOLED = 1, VP_WKIND_UPSAMPLED = 2 };
enum { VP_WLAYOUT_FWD = 0, VP_WLAYOUT_DGRAD = 1,
       VP_WLAYOUT_RESIDUAL = 4 /* OR-ed in: pack tf32(w - tf32(w)), the low part of the fp32-exact 3xTF32 mode */ };

const char* vp_last_error(void);
/* debug: per-CTA globaltimer stamps of the last vp_conv_igemm launch made with VP_FWD_TRACE=1 (8 x u64 per CTA) */
int vp_debug_read_trace(unsigned long long* host, int n_ctas);
int vp_version(void);

/* ---- tensor-core implicit-GEMM convolution (tcgen05 / TMEM / TMA) ------------------------------
 * Replaces tf.nn.conv2d (rnn_ops.py:121, ops.py:528), tf.nn.conv2d_transpose (ops.py:584),
 * tf.nn.conv3d (ops.py:773) and their gradients.
 * wpacked: [kd*kh*kw][n_pad][kc*32] floats (see vp_pack_weights); GEMM N = n_pad (multiple of 16),
 * GEMM K = kc 32-channel chunks of in->c per tap.  out->c columns are stored.
 * split_k > 1: partial sums are atomically added into `out` (caller zero-fills, or leaves the prior of accumulate = 1 / 2
 * in place; act must be NONE; bias is added by split 0).  split_k == 0: automatic -- an under-filled grid with a long K loop is split and a DENSE
 * output (out->c == out->cstride) is cleared by the call itself.  accumulate = 1: out += result (act must be NONE);
 * accumulate = 2: out = act(out + result + bias) -- the last pass of a multi-pass (3xTF32) accumulation. */
int vp_conv_igemm(const vp_tensor* in, const vp_conv_geom* g, const float* wpacked, int n_pad, int kc,
                  const vp_tensor* out, const float* bias, int act, float alpha, int split_k, int accumulate,
                  vp_stream_t stream);

/* Engine selection for vp_conv_igemm / vp_conv_igemm_actgrad on the calling thread: 0 = box mode (one activation tile per
 * filter tap), 1 = halo mode (one halo tile per tap group, 256 output positions per CTA; falls back to box mode when the
 * geometry is not eligible), -1 = default (halo unless the environment says VP_HALO=0).  Both engines compute the same
 * sums (fp32 summation order differs); the host layer times both once per geometry and keeps the faster. */
int vp_conv_set_engine(int engine);

/* What the calling thread's last vp_conv_igemm / vp_conv_igemm_actgrad / vp_conv_wgrad call launched: info[0] = kernel
 * (0 = box mode, 1 = halo mode, 2 = weight gradient by tap groups, 3 = weight gradient by rows; -1 = none yet),
 * info[1] = the number of K splits it ran with.  Lets a caller see which path served a call (halo mode falls back to box
 * mode on ineligible geometries, split_k = 0 chooses the splits). */
int vp_conv_last_launch(int* info);

/* Input-gradient convolution fused with the backward of the previous layer's activation:
 *   out = (conv(in) + addend) * act'(act_output),  act' evaluated from the activation OUTPUT (lrelu/relu/sigmoid/tanh);
 * act_output / addend (optional) have exactly the layout of the dense `out`.  Used for the discriminator towers
 * (lrelu(conv3d), networks.py:83-102), where it removes one full read+write pass per layer. */
int vp_conv_igemm_actgrad(const vp_tensor* in, const vp_conv_geom* g, const float* wpacked, int n_pad, int kc,
                          const vp_tensor* out, const float* act_output, const float* addend, int act, float alpha,
                          int accumulate /* 0, or 2: the existing `out` is added to conv(in) first */, vp_stream_t stream);

/* lo = x - tf32_truncate(x) over n floats (16-byte aligned, n % 4 == 0): the part of an fp32 activation the tensor core
 * does not read.  conv(x, W) + conv(lo, W) + conv(x, W_residual) is the fp32-exact ("3xTF32") debug mode. */
int vp_tf32_residual(const float* x, float* lo, long long n, vp_stream_t stream);

/* Weight gradient of the same convolution: dwpacked[tap][co][ci] += sum_o  dy.. * x..
 * (layout VP_WLAYOUT_FWD: rows = channels of dy (n_pad rows), cols = kc*32 channels of x).
 * Always accumulates atomically: caller zero-fills before the first call of a step. */
int vp_conv_wgrad(const vp_tensor* x, const vp_tensor* dy, const vp_conv_geom* g, float* dwpacked, int n_pad,
                  int kc, int split_k, vp_stream_t stream);

/* Weight packing: reference-layout kernel w [kd][kh][kw][ci_ref][co] (HWIO / DHWIO) ->
 * effective tap matrices in tensor-core layout, TF32-rounded.
 *  kind PLAIN:     taps = kd*kh*kw, Keff = w
 *  kind POOLED:    2-D only, taps = (kh+1)*(kw+1): avg-pool(2x2,s1,FULL) of the kernel (ops.py:838-842)
 *  kind UPSAMPLED: 2-D only, taps = (kh+3)*(kw+3): bilinear (x) kernel (ops.py:698-704)
 *  layout FWD:   wpacked[tap][co (n_pad)][ci_int (kc*32)]
 *  layout DGRAD: wpacked[tap][ci_int (n_pad)][co (kc*32)]
 * cmap[ci_int] = reference input channel feeding internal channel ci_int, or -1 (zero column);
 * cmap == NULL means identity.  inv_scale: optional device scalar; weights are divided by it
 * (spectral norm sigma, ops.py:1044). */
int vp_pack_weights(const float* w, int kd, int kh, int kw, int ci_ref, int co, int kind, int layout,
                    const int32_t* cmap, int ci_int, const float* inv_scale, float* wpacked, int n_pad, int kc,
                    vp_stream_t stream);
/* The same for a whole table of tensors in one launch.  `jobs_device` is a DEVICE array; job i owns the 256-thread blocks
 * [block_begin_i, block_begin_{i+1}) with block_begin_0 = 0 and ceil(taps * n_pad * kc * 32 / 256) blocks per job;
 * total_blocks = the sum.  Fields as the arguments of vp_pack_weights. */
typedef struct {
  const float* w;
  float* wpacked;
  const int32_t* cmap;
  const float* inv_scale;
  int kd, kh, kw, ci_ref, co, kind, layout, ci_int, n_pad, kc;
  int block_begin;
  int reserved;
} vp_pack_job;
int vp_pack_weights_batch(const vp_pack_job* jobs_device, int njobs, int total_blocks, vp_stream_t stream);
/* Adjoint of vp_pack_weights(layout FWD): dw[...] += L^T(dwpacked) (no scale applied). */
int vp_unpack_wgrad(const float* dwpacked, int kd, int kh, int kw, int ci_ref, int co, int kind,
                    const int32_t* cmap, int ci_int, float* dw, int n_pad, int kc, vp_stream_t stream);


/* ---- HBM-bound kernels --------------------------------------------------------------------------
 * "positions" = product of the spatial dims of one sample; x[(n*positions + p)*cstride + ch]. */

/* fused_instance_norm (+ activation), layers/normalization.py:34-196 + savp_model.py:463-464:
 * y = act(gamma*(x-mean)*rsqrt(var_biased+eps)+beta), stats over `positions` per (sample, channel).
 * stats (optional): [n][c][2] = (mean, rstd) kept for the backward pass. c % 4 == 0. */
int vp_inorm_act(const float* x, int x_cstride, float* y, int y_cstride, int n, int positions, int c,
                 const float* gamma, const float* beta, float eps, int act, float alpha, float* stats,
                 vp_stream_t stream);

/* BasicConv2DLSTMCell gate math, rnn_ops.py:148-165 (instance norm over the 4F concat, i/j/f/o
 * split, forget bias, instance norm of new_c, h = tanh(c)*sigmoid(o)).  pre: conv output
 * [n][positions][4*filters] dense; c_prev/c_new: [n][positions][filters] dense.  h is written to
 * num_h_dst (1..3) channel slices h_dst[i] with channel strides h_cstride[i].
 * stats1 [n][4F][2], stats2 [n][F][2] optional. positions <= 1024, filters % 4 == 0. */
int vp_lstm_gates_fwd(const float* pre, int n, int positions, int filters, const float* c_prev,
                      const float* gamma1, const float* beta1, const float* gamma2, const float* beta2,
                      float forget_bias, float eps, float* c_new, float* const* h_dst, const int* h_cstride,
                      int num_h_dst, float* stats1, float* stats2, vp_stream_t stream);

/* ops.tile_concat (ops.py:968-1006): dst[n][p][0..c) = vec[n][0..c) for every position p. */
int vp_broadcast_channels(const float* vec, int vec_stride, float* dst, int dst_cstride, int n, int positions,
                          int c, vp_stream_t stream);
/* channel-slice copy: dst[r][0..c) = src[r][0..c) for r < rows. */
int vp_copy_channels(const float* src, int src_cstride, float* dst, int dst_cstride, long long rows, int c,
                     vp_stream_t stream);
/* tf.where(ground_truth[t], images, gen_image) (savp_model.py:406): out[i] = sel[i] ? a[i] : b[i], rows of per_row floats. */
int vp_select_rows(const int32_t* sel, const float* a, const float* b, float* out, int n, long long per_row,
                   vp_stream_t stream);
/* global average pool (networks.py:30-31): y[n][c] = mean_p x[n][p][c]. */
int vp_avgpool(const float* x, int x_cstride, float* y, int n, int positions, int c, vp_stream_t stream);
/* ops.dense (ops.py:5-16): y[b][j] = sum_k x[b][k] w[k][j] / (*inv_scale) + bias[j].
 * k_splits > 1 accumulates atomically into a zero-filled y. */
int vp_dense_fwd(const float* x, int x_stride, const float* w, const float* bias, const float* inv_scale, float* y,
                 int y_stride, int b, int k, int j, int k_splits, vp_stream_t stream);
/* tf.nn.rnn_cell.LSTMCell elementwise part (savp_model.py:354-362); gates [b][4*units] (i,j,f,o). */
int vp_lstm_cell_fwd(const float* gates, const float* c_prev, float* c_new, float* h_new, int b, int units,
                     float forget_bias, vp_stream_t stream);
/* savp_model.py:49,712: lss <- clip(lss,-10,10); z = mu + sqrt(exp(lss))*eps. */
int vp_sample_z(const float* mu, float* log_sigma_sq, const float* eps, float* z, int total, vp_stream_t stream);
/* savp_model.py:551-559: +identity kernel, relu(.-1e-12)+1e-12, normalise over the kh*kw taps.
 * raw/out: [b][kh*kw][nk]. */
int vp_cdna_kernel_norm(const float* raw, float* out, int b, int kh, int kw, int nk, vp_stream_t stream);
/* apply_cdna_kernels (savp_model.py:893-923) + the two background layers (:581-584): image and
 * first_image are [n][h][w][4] (colour channels padded to 4); writes nk+2 float4 slots per pixel at
 * layers[(n*h*w+p)*layers_cstride + 4*l]. */
int vp_cdna_apply(const float* image, const float* first_image, const float* kernels, float* layers,
                  int layers_cstride, int n, int h, int w, int kh, int kw, int nk, vp_stream_t stream);
/* flow_ops.image_warp (flow_ops.py:4-79; transformation='flow', savp_model.py:955-965): backward bilinear warp with
 * the neighbour indices clipped to the image; flow [n][h][w][2] = (x, y) displacement.  bwd: dim += (atomic, may be
 * NULL), dflow overwritten (may be NULL). */
int vp_image_warp_fwd(const float* im, int im_cstride, const float* flow, float* out, int out_cstride, int n, int h, int w,
                      int c, vp_stream_t stream);
int vp_image_warp_bwd(const float* im, int im_cstride, const float* flow, const float* dout, int dout_cstride, float* dim,
                      int dim_cstride, float* dflow, int n, int h, int w, int c, vp_stream_t stream);
/* masks = softmax(logits) (savp_model.py:634); gen_image = sum_l layer_l * mask_l (:645-646). */
int vp_composite(const float* logits, int logits_cstride, const float* layers, int layers_cstride, float* masks,
                 int masks_cstride, float* gen_image, long long positions, int num_layers, vp_stream_t stream);


/* ---- backward passes of the HBM-bound kernels ----------------------------------------------------
 * Gradient inputs that have several consumers are passed as lists of (pointer, channel stride)
 * "sources" which the kernel sums.  Parameter gradients (dgamma, dbeta, dw, db ...) are ACCUMULATED. */
int vp_inorm_act_bwd(const float* x, int x_cstride, const float* const* dy, const int* dy_cstride, int num_dy,
                     float* dx, int dx_cstride, int n, int positions, int c, const float* gamma, const float* beta,
                     const float* stats, int act, float alpha, float* dgamma, float* dbeta, vp_stream_t stream);
int vp_lstm_gates_bwd(const float* pre, int n, int positions, int filters, const float* c_prev, const float* gamma1,
                      const float* beta1, const float* gamma2, const float* beta2, const float* stats1,
                      const float* stats2, float forget_bias, const float* const* dh, const int* dh_cstride,
                      int num_dh, const float* dc_next, float* dpre, float* dc_prev, float* dgamma1, float* dbeta1,
                      float* dgamma2, float* dbeta2, vp_stream_t stream);
int vp_composite_bwd(const float* dgen, const float* masks, int masks_cstride, const float* layers, int layers_cstride,
                     float* dlogits, int dlogits_cstride, float* dlayers, int dlayers_cstride, long long positions,
                     int num_layers, vp_stream_t stream);
/* dT_k = d_a[..,4k] + d_b[..,4k]; dimage += (atomic) ; dkernels += (atomic) */
int vp_cdna_apply_bwd(const float* image, const float* kernels, const float* d_a, int d_a_cstride, const float* d_b,
                      int d_b_cstride, float* dimage, float* dkernels, int n, int h, int w, int kh, int kw, int nk,
                      vp_stream_t stream);
int vp_cdna_kernel_norm_bwd(const float* raw, const float* out, const float* dout, float* draw, int b, int kh, int kw,
                            int nk, vp_stream_t stream);
/* dx (optional; overwritten or accumulated), dw += , dbias += */
int vp_dense_bwd(const float* x, int x_stride, const float* w, const float* inv_scale, const float* dy, int dy_stride,
                 float* dx, int dx_stride, int dx_accumulate, float* dw, float* dbias, int b, int k, int j,
                 vp_stream_t stream);
int vp_lstm_cell_bwd(const float* gates, const float* c_prev, const float* c_new, const float* dh, const float* dc_next,
                     float* dgates, float* dc_prev, int b, int units, float forget_bias, vp_stream_t stream);
/* out[n*out_stride + c] += scale * sum_p x[n][p][c] */
int vp_colsum(const float* x, int x_cstride, float* out, int out_stride, int n, long long positions, int c, float scale,
              vp_stream_t stream);
/* dst[r][c] = (accumulate ? dst[r][c] : 0) + scale*src[r][c]; rows whose row_mask[r / rows_per_mask] != 0 contribute 0 */
int vp_axpy_channels(const float* src, int src_cstride, float* dst, int dst_cstride, long long rows, int c, float scale,
                     const int32_t* row_mask, long long rows_per_mask, int accumulate, vp_stream_t stream);
/* dx = (dy_a + dy_b) * act'(.) evaluated from the activation OUTPUT y */
int vp_act_bwd(const float* y, int y_cstride, const float* dy_a, int dy_a_cstride, const float* dy_b, int dy_b_cstride,
               float* dx, int dx_cstride, long long rows, int c, int act, float alpha, vp_stream_t stream);
int vp_avgpool_bwd(const float* dy, float* dx, int dx_cstride, int n, int positions, int c, vp_stream_t stream);
/* *kl_scale (device scalar, may be NULL = 0) = kl_weight(step) / rows, rows = (T-1)*B; dz may be NULL */
int vp_sample_z_bwd(const float* mu, const float* lss, const float* eps, const float* dz, float* dmu, float* dlss,
                    int total, const float* kl_scale, vp_stream_t stream);

/* transformation = 'flow' (savp_model.py:522-530, 577-578; flow_ops.image_warp, flow_ops.py:4-79; apply_flows, :955-965):
 * NK backward bilinear warps of `image` (float4 pixels) by the flows-conv output [N,H,W,flows_cstride] (channel k = x-flow of
 * transform k, channel NK + k = y-flow), written with the previous and the first image as float4 slots 0..NK+1 of `layers`
 * (the slot layout of vp_cdna_apply).  Backward: dimage += (zero-filled by the caller), dflows = (same layout as flows). */
int vp_flow_apply(const float* image, const float* first_image, const float* flows, int flows_cstride, float* layers,
                  int layers_cstride, int n, int h, int w, int nk, vp_stream_t stream);
int vp_flow_apply_bwd(const float* image, const float* flows, int flows_cstride, const float* d_a, int d_a_cstride,
                      const float* d_b, int d_b_cstride, float* dimage, float* dflows, int n, int h, int w, int nk,
                      vp_stream_t stream);

/* ---- losses (losses.py:6-67): out[0] += value; optional gradient = grad_scale * d value / d pred -------- */
int vp_pixel_loss(const float* pred, int pred_cstride, const float* target, int target_cstride, float* dpred,
                  int dpred_cstride, long long rows, int c, int mode /*bit 0: 0 = L1, 1 = L2; bit 1: dpred += instead of =*/, long long mean_count,
                  float grad_scale, float* out, vp_stream_t stream);
/* losses.gan_loss (losses.py:29-54) for labels in {0,1}: kind 0 LSGAN, 1 GAN (sigmoid cross-entropy), 2 SNGAN (softplus) */
int vp_gan_loss(const float* logits, float label, int n, float grad_scale, int kind, float* dlogits, float* out,
                vp_stream_t stream);
int vp_kl_loss(const float* mu, const float* lss, int rows, int nz, float* out, vp_stream_t stream);
/* cosine_distance(a, b) over rows of c channels; da += grad (gradient w.r.t. a only) */
int vp_cosine_distance(const float* a, const float* b, float* da, long long rows, int c, float grad_scale, float* out,
                       vp_stream_t stream);
/* tf.train.AdamOptimizer (TF1 epsilon-hat form).  *lr_t (device scalar) = lr*sqrt(1-beta2^t)/(1-beta1^t): step-dependent
 * scalars live in device memory so that a captured CUDA graph of the step stays valid.  g is multiplied by grad_scale. */
int vp_adam(float* p, const float* g, float* m, float* v, long long n, const float* lr_t, float beta1, float beta2,
            float eps, float grad_scale, vp_stream_t stream);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
long long vp_launch_count(void);

/* ---- discriminator helpers ------------------------------------------------------------------------
 * spectral_normed_weight (ops.py:1020-1049): w [rows][cols] (rows = prod(kernel dims)*cin), u [cols].
 * fwd: v [rows] = l2n(W u), s [cols] = v W, u_new = l2n(s), scal[0..2] = (|Wu|, |s|, sigma).
 * bwd: dw += d(W/sigma)/dW applied to g_wbar, differentiating through the power iteration;
 *      gs [cols], gt [rows] are scratch; scal[3] is scratch. */
int vp_spectral_norm_fwd(const float* w, const float* u, int rows, int cols, float* v, float* s, float* u_new,
                         float* scal, vp_stream_t stream);
int vp_spectral_norm_bwd(const float* w, const float* u, const float* g_wbar, int rows, int cols, const float* v,
                         const float* s, float* scal, float* gs, float* gt, float* dw, vp_stream_t stream);
/* First discriminator layer on the CUDA cores (conv3d 3x3x3, stride 1, zero pad 1, <= 4 input channels stored as
 * float4 voxels, 32 output channels, fused bias + leaky relu; networks.py:83-84).  w is the REFERENCE-layout kernel
 * [3][3][3][ci][32]; it is divided by *inv_scale (spectral-norm sigma).  wgrad accumulates dL/d(w/sigma) into gw. */
int vp_conv3d_c4_fwd(const float* x, const float* w, const float* inv_scale, const float* bias, float* out, int n, int d,
                     int h, int wd, int ci, float lrelu_alpha, vp_stream_t stream);
int vp_conv3d_c4_wgrad(const float* x, const float* dy, float* gw, int n, int d, int h, int wd, int ci, vp_stream_t stream);
/* The same layer on the tensor cores (TF32 operands, fp32 accumulate), without repacking x (csrc/d0_layer.cu):
 *  fwd:   a flat halo tile of float4 voxels is the un-swizzled K-major operand; the next-voxel leading offset (LBO = 16 B)
 *         turns x[v-1 .. v+2] into the K = 16 operand of one kernel row.  Needs h % 4 == 0 and a tile that fits (64^2, 128^2 do).
 *  wgrad: rows of float4 voxels are the 32-byte-atom MN-major operand, dy arrives phase-major.  Needs wd % 64 == 0. */
int vp_conv3d_c4_fwd_tc(const float* x, const float* w, const float* inv_scale, const float* bias, float* out, int n, int d, int h,
                        int wd, int ci, float lrelu_alpha, vp_stream_t stream);
int vp_conv3d_c4_wgrad_tc(const float* x, const float* dy, float* gw, int n, int d, int h, int wd, int ci, vp_stream_t stream);
/* savp_model.py:97-102: clip[b][j][p] = video[t_start[b]+j][batch_offset+b][p]; pixels = H*W (4 floats each) */
int vp_gather_clip(const float* video, const int32_t* t_start, float* clip, int clips, int clip_len, long long pixels,
                   int video_batch, int batch_offset, vp_stream_t stream);
int vp_scatter_clip(const float* dclip, const int32_t* t_start, float* dvideo, int clips, int clip_len, long long pixels,
                    int video_batch, int batch_offset, vp_stream_t stream);

/* Debug: one tcgen05.mma kind::tf32 (M = 128, N = n, K = 8) on caller-supplied shared-memory images and descriptor fields
 * (start offset, LBO, SBO in bytes; layout type 0 none, 1 = 128B/32B-atom, 2 = 128B; major 0 = K, 1 = MN).  out = [128][n]. */
int vp_debug_umma_probe(const void* a_img, int a_bytes, const void* b_img, int b_bytes, unsigned a_start, unsigned a_lbo,
                        unsigned a_sbo, unsigned a_layout, int a_mn_major, unsigned b_start, unsigned b_lbo, unsigned b_sbo,
                        unsigned b_layout, int b_mn_major, int n, float* out, vp_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* VP_B200_H_ */
