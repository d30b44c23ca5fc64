/* trainner_b200 -- C ABI of the B200-native ESRGAN hot path (sm_100a).
 *
 * Drop-in boundary for the library calls the reference makes on its G/D training step
 * (paths relative to victorca25/traiNNer codes/):
 *   nn.Conv2d fwd / autograd dgrad / wgrad   models/modules/architectures/block.py:238
 *   torch.cat + LeakyReLU + 0.2*x5+x          architectures/RRDBNet_arch.py:150-163 (fused epilogues)
 *   F.interpolate(nearest x2)                 architectures/block.py:358         (store-replicate epilogue)
 *   nn.BatchNorm2d (train)                    architectures/block.py:122
 *   nn.MaxPool2d / ReLU / input-norm          architectures/perceptual.py:152-214
 *   nn.L1Loss                                 models/losses.py:37-39
 *
 * Conventions: all pointers are DEVICE pointers owned by the caller (PyTorch allocator); the
 * library never frees or retains them past the call.  Activations are NHWC bf16; images that
 * cross the nn.Module boundary are NCHW fp32.  Every call enqueues on `stream` and returns
 * without synchronising.  Return value 0 = ok, nonzero = error; message via
 * b200_last_error() (thread-local).  No CPU fallback exists: on a machine without an sm_100
 * device every compute entry point returns an error.
 */
#ifndef TRAINNER_B200_H_
#define TRAINNER_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* b200_stream_t; /* cudaStream_t */

#define B200_MAX_TAPS 16

/* Implicit-GEMM convolution on tcgen05 tensor cores.  One descriptor covers fwd, dgrad
 * (with weights packed [tap][ci][co]) and the parity-decomposed dgrad of stride-2 convs.
 *   out[n, y*out_mul_y+out_off_y, x*out_mul_x+out_off_x, cout_off + co] = epilogue(
 *       sum_t sum_ci in[n, y*in_stride+in_off_y+tap_dy[t], x*in_stride+in_off_x+tap_dx[t], cin_off+ci]
 *                    * w[tap_w[t]][co][ci] )
 * epilogue(v): v = alpha*(v + bias[co]) (+beta1*res1) (+beta2*res2) (+old out if accumulate)
 *              -> lrelu(slope) if act -> times lrelu'(mask) for co in [mask_lo, mask_hi).     */
typedef struct {
  int32_t n, h_in, w_in;        /* input tensor [n, h_in, w_in, cx]                         */
  int32_t cx, cin_off, cin;     /* input channel slice; cin % 16 == 0                       */
  int32_t h_out, w_out;         /* logical output grid (before placement)                   */
  int32_t h_buf, w_buf, cy;     /* output tensor [n, h_buf, w_buf, cy]                      */
  int32_t cout_off, cout;       /* output channel slice; cout % 8 == 0                      */
  int32_t ntaps;
  int8_t tap_dy[B200_MAX_TAPS], tap_dx[B200_MAX_TAPS], tap_w[B200_MAX_TAPS];
  int32_t in_stride, in_off_y, in_off_x;
  int32_t out_mul_y, out_off_y, out_mul_x, out_off_x;
  int32_t upsample2x;           /* 1: replicate every output to a 2x2 block (h_buf = 2*h_out) */
  int32_t w_taps, w_cout_pad, w_cin_pad; /* packed weights [w_taps][w_cout_pad][w_cin_pad] bf16 */
  float alpha;
  int32_t act;                  /* 0 none, 1 leaky-relu(slope) (slope 0 = relu)             */
  float slope;
  float beta1, beta2;
  int32_t res_nch;              /* residuals apply to co < res_nch                          */
  int32_t res1_c, res1_coff, res2_c, res2_coff; /* res tensors [n, h_buf, w_buf, res_c] ([n,h_out,w_out,.] if upsample2x) */
  int32_t accumulate;
  int32_t mask_c, mask_coff, mask_lo, mask_hi;  /* mask tensor [n, h_buf, w_buf, mask_c]     */
  float mask_slope;
  /* 4: ONE launch computes the four output-parity classes of the dgrad of a 4x4 stride-2 conv: class c uses taps
   * [c*ntaps, (c+1)*ntaps) of the tap tables and writes at out_off + (c >> 1, c & 1) (out_mul must be (2,2)).
   * 0 / 1: a single conv. */
  int32_t parity_classes;
} b200_conv_desc;

int b200_conv_igemm(const b200_conv_desc* d, const void* x, const void* w_packed, const float* bias,
                    const void* res1, const void* res2, const void* mask, void* y,
                    b200_stream_t stream);
/* The same conv (no residual / mask / activation operands) that ALSO writes the BatchNorm partial statistics of
 * its bf16-rounded output from the epilogue: stat_part is fp32 [2][cout][rows], rows = b200_conv_igemm_stat_rows(d)
 * (0 when this shape is not served by the statistics epilogue -- use b200_bn_stats_finalize then; < 0 on error).
 * Replaces the separate pass of nn.BatchNorm2d's batch statistics over the conv output (block.py:122).        */
int b200_conv_igemm_stat_rows(const b200_conv_desc* d);
int b200_conv_igemm_stats(const b200_conv_desc* d, const void* x, const void* w_packed, const float* bias,
                          void* y, float* stat_part, b200_stream_t stream);

/* 3x3 stride-1 pad-1 convolution on ZERO-BORDERED ("flat") activations, the trunk fast path.
 * Tensors are [n, h+2, w+2, c] NHWC bf16 whose 1-pixel border is zero and never written; with the
 * border in place a tap is a pure row shift of the flattened [n*(h+2)*(w+2), c] matrix, so one
 * haloed smem tile serves all 9 taps (9x less L2->SMEM traffic than per-tap loading):
 *   out[m, cout_off+co] = epilogue( sum_t sum_ci in[m + tap_shift(t), cin_off+ci] * w[tap_w[t]][co][ci] )
 * for interior positions m only.  tap_shift(t) = tap_dy[t]*(w+2) + tap_dx[t].  Epilogue as in
 * b200_conv_igemm; res1/res2/mask are flat tensors indexed by the same m.
 * out_mode 0: flat output [n,h+2,w+2,cy]; 1: dense [n,h,w,cy]; 2: dense with 2x2 replication
 * [n,2h,2w,cy] (nearest upsample folded into the store).                                      */
typedef struct {
  int32_t n, h, w;              /* interior size; buffers are (h+2) x (w+2)                  */
  int32_t cx, cin_off, cin;
  int32_t cx2, cin2_off, cin2;  /* optional second input (flat, same grid): its channels extend the
                                   reduction axis after the first input's (cin padded to 64)     */
  int32_t cy, cout_off, cout;   /* cout % 16 == 0, cout <= 192                               */
  int8_t tap_dy[9], tap_dx[9], tap_w[9];
  int32_t out_mode;
  int32_t w_taps, w_cout_pad, w_cin_pad;
  float alpha;
  int32_t act;
  float slope;
  float beta1, beta2;
  int32_t res_nch, res1_c, res1_coff, res2_c, res2_coff;
  int32_t accumulate;
  int32_t mask_c, mask_coff, mask_lo, mask_hi;
  float mask_slope;
} b200_flat_desc;

int b200_conv3x3_flat(const b200_flat_desc* d, const void* x, const void* x2, const void* w_packed,
                      const float* bias, const void* res1, const void* res2, const void* mask, void* y,
                      b200_stream_t stream);

/* layout helpers between dense [n,h,w,c] and flat [n,h+2,w+2,c] slices (bf16):
 * pad_copy:  flat[interior, dst_coff + c] = dense[.., src_coff + c]
 * unpad_add: dense[.., c] = flat[interior, src_coff + c] (+ add[.., c] when add != NULL)       */
int b200_pad_copy(void* dst_flat, int32_t dst_c, int32_t dst_coff, const void* src_dense, int32_t src_c,
                  int32_t src_coff, int32_t n, int32_t h, int32_t w, int32_t c, b200_stream_t stream);
int b200_unpad_add(void* dst_dense, int32_t dst_c, const void* src_flat, int32_t src_c, int32_t src_coff,
                   const void* add_dense, int32_t add_c, int32_t n, int32_t h, int32_t w, int32_t c,
                   b200_stream_t stream);

/* Whole-trunk chain of dense blocks in ONE persistent launch (csrc/rdb_chain.cu).  A block is computed input
 * slice by input slice: stage j adds the newest slice's contribution to every conv that still needs it, with the
 * fp32 partial sums of a CTA's 256-position super-tile kept in TMEM for the whole block, and the slice each stage
 * completes is kept in shared memory as the next stage's operand.  One CTA per super-tile, all co-resident; halo
 * rows travel between neighbouring CTAs of a thread-block cluster through distributed shared memory and across
 * cluster edges through L2 in flag-in-data (LL) form.  Replaces the 5 x n_blocks per-conv launches of
 * ResidualDenseBlock_5C.forward / RRDB.forward (RRDBNet_arch.py:89-96,150-163) and of their input gradients.  Stage s = 5*block + j: input slice = the output slice of stage s-1 (stage 0:
 * channels [x_coff, x_coff+64) of x0), epilogue
 *   v = alpha*(acc + bias) + beta1*res1 + beta2*res2 ; act ? lrelu(v, slope) ; mask ? (mask > 0 ? v : mask_slope*v)
 * for the 32 (j = 4: 64) channels that stage completes, stored to out[m*out_c + out_coff ..] (bf16, interior
 * positions only; NULL = not stored).  All tensors are flat zero-bordered [n_total, h+2, w+2, C] bf16. */
typedef struct {
  void* out;
  const float* bias;     /* indexed by channel within the stage's completing slice, or NULL */
  const void* mask;
  const void* res1;
  const void* res2;
  int32_t out_c, out_coff, mask_c, mask_coff, res1_c, res1_coff, res2_c, res2_coff;
  float alpha, beta1, beta2, slope, mask_slope;
  int32_t act;
  int32_t pad_[2];
} b200_chain_stage;

typedef struct {
  int32_t n_total, img0, n;   /* images in the tensors; first image and image count of this launch */
  int32_t h, w;
  int32_t cx, x_coff;         /* channel pitch / offset of the first block's 64-channel input in x0 */
  int32_t n_blocks;
  int32_t flip_taps;          /* 0: forward taps; 1: input-gradient taps */
} b200_chain_desc;

/* CTAs (= 256-position super-tiles; must not exceed the SM count) and exchange-buffer bytes for n images;
 * returns nonzero when the image is too wide for the kernel (w > 125) */
int b200_rdb_chain_geometry(int32_t n, int32_t h, int32_t w, int32_t* n_cta, int64_t* ll_bytes);
/* w_stage[j]: packed stage weights [n_blocks][9][192-32j][K_j] bf16 (K_0 = 64, K_j = 32); table_dev:
 * [n_blocks][5] b200_chain_stage in device memory; ll_buf: zero-initialised once, reused by every launch;
 * epoch_dev: one uint32 in device memory (zero-initialised), owned by the library between launches. */
int b200_rdb_chain(const b200_chain_desc* d, const void* x0, const void* const* w_stage,
                   const b200_chain_stage* table_dev, void* ll_buf, int64_t ll_bytes, uint32_t* epoch_dev,
                   b200_stream_t stream);

/* Weight gradient of a conv (autograd wgrad of block.py:238):
 *   dw[co][ci][ky][kx] += scale * sum_{n,y,x} dy[n,y,x,dy_coff+co] * x[n, y*stride+ky-pad, x*stride+kx-pad, x_coff+ci]
 * dw is fp32 OIHW (the layout of nn.Conv2d.weight.grad); accumulated with fp32 atomics.      */
typedef struct {
  int32_t n, h_in, w_in, cx, x_coff, cin;
  int32_t h_out, w_out, cdy, dy_coff, cout;
  int32_t kh, kw, stride, pad;
  float scale;
} b200_wgrad_desc;

int b200_conv_wgrad(const b200_wgrad_desc* d, const void* x, const void* dy, float* dw,
                    float* dbias, b200_stream_t stream);

/* Weight gradients of ALL residual dense blocks in one launch (flat layout, nf = 64, gc = 32).
 * Per block r: x = B[r] [P,192], g = G[r] (conv1..4 pre-activation grads in channels 64..191),
 * dO = G[r+1][:, 0:64] (conv5's dY up to scale5).  dw[k] are the fp32 OIHW gradient tensors of
 * conv1..conv5 (accumulated with +=).  Tensor maps are encoded on the host into `maps_host`
 * (3 * n_rdb * b200_tensor_map_bytes() bytes, 64-byte aligned) and copied to the device by the caller. */
typedef struct {
  float* dw[5];
  float scale5;
  int32_t pad_;
} b200_wgrad_rdb_entry;

int b200_tensor_map_bytes(void);
int b200_wgrad_rdb_make_maps(void* maps_host, int32_t n_rdb, const void* const* x_ptrs,
                             const void* const* g_ptrs, const void* const* do_ptrs,
                             const int32_t* do_pitch, int32_t n, int32_t h, int32_t w, int32_t c);
/* The positions are reduced in slices (L2 locality); each slice parks its partial sums in a caller-provided
 * workspace of b200_wgrad_rdb_ws_bytes() bytes and a second kernel adds the slices in a fixed order
 * (deterministic: no float atomics). */
int64_t b200_wgrad_rdb_ws_bytes(int32_t n_rdb, int32_t n, int32_t h, int32_t w);
int b200_wgrad_rdb(const void* maps_dev, const b200_wgrad_rdb_entry* entries_dev, int32_t n_rdb,
                   int32_t n, int32_t h, int32_t w, int32_t nf, int32_t gc, void* workspace,
                   int64_t ws_bytes, b200_stream_t stream);

/* Many per-channel column sums in one launch: dst[c] += scale * sum_p src[p*pitch + coff + c]  (bias grads) */
typedef struct {
  const void* src;   /* bf16 */
  float* dst;
  int64_t npix;
  int32_t pitch, coff, c;
  float scale;
} b200_colsum_entry;

int b200_colsum_multi(const b200_colsum_entry* table_dev, int32_t count, b200_stream_t stream);

/* Pack fp32 OIHW conv weights into the bf16 tensor-core layouts, many tensors per launch.
 * table: device array of b200_pack_entry.  mode 0: [tap][co][ci] (fwd); 1: [tap][ci][co] (dgrad) */
typedef struct {
  const float* src;  /* [cout][cin][kh*kw] */
  void* dst;         /* bf16 [taps][rows_pad][cols_pad] */
  int32_t cout, cin, taps, rows_pad, cols_pad, mode;
  int32_t co_mul, co_off; /* source output channel = co * co_mul + co_off (pixel-shuffle groups); 0,0 = identity */
} b200_pack_entry;

int b200_pack_weights(const b200_pack_entry* table_dev, int32_t count, int32_t max_elems,
                      b200_stream_t stream);

/* Pack a block of an fp32 OIHW weight into a column range of a concatenated dgrad matrix
 * dst[tap][row][col_off + co] = scale * src[co][ci_off + row][tap] for row < n_rows, co < cout
 * (dst is bf16 [taps][rows_pad][cols_pad], zero-initialised once by the caller).  Used by the
 * gather form of the RDB input gradient: one GEMM per channel slice over all later convs.     */
typedef struct {
  const float* src;
  void* dst;
  int32_t cout, cin, taps, ci_off, n_rows, rows_pad, cols_pad, col_off;
  float scale;
  int32_t row_off;  /* destination row offset */
  int32_t mode;     /* 1 (default 0 means 1 for backward compatibility is NOT applied): see below */
  int32_t pad_;
} b200_packcat_entry;
/* mode 1: rows = input channels : dst[t][row_off + r][col_off + co] = scale*src[co][ci_off + r][t], r < n_rows
 * mode 0: rows = output channels: dst[t][row_off + co][col_off + c] = scale*src[co][ci_off + c][t], c < n_rows */

int b200_pack_cat(const b200_packcat_entry* table_dev, int32_t count, int32_t max_elems,
                  b200_stream_t stream);

/* 3x3 stride-1 pad-1 convolutions with a thin (<= 4 channel) side, CUDA-core direct kernels.
 * thin->wide: x NCHW fp32 [n,cs,h,w] -> y NHWC bf16 [n,h,w,cy] slice, optional per-channel input
 *             normalisation (x-mean)/std (perceptual.py:207) and lrelu/relu epilogue.
 * wide->thin: x NHWC bf16 -> y NCHW fp32 [n,cs,h,w] (+bias).                                   */
int b200_conv3x3_thin_to_wide(const float* x, const float* w_oihw, const float* bias, void* y,
                              int32_t n, int32_t h, int32_t w, int32_t cs, int32_t cw, int32_t cy,
                              int32_t y_coff, int32_t transpose_w, const float* mean,
                              const float* std, int32_t act, float slope, const void* mask,
                              int32_t mask_c, int32_t mask_coff, float mask_slope,
                              b200_stream_t stream);
int b200_conv3x3_wide_to_thin(const void* x, const float* w_oihw, const float* bias, float* y,
                              int32_t n, int32_t h, int32_t w, int32_t cw, int32_t cx, int32_t x_coff,
                              int32_t cs, int32_t transpose_w, const float* inv_std, float out_scale,
                              b200_stream_t stream);
/* wgrad of either: dw[cw_idx][cs_idx][3][3] (thin side fp32 NCHW, wide side bf16 NHWC).
 * wide_is_out = 1: dw is [cw][cs][3][3] (thin->wide conv); 0: dw is [cs][cw][3][3].          */
int b200_conv3x3_thin_wgrad(const float* thin, const void* wide, float* dw, float* dbias_wide,
                            float* dbias_thin, int32_t n, int32_t h, int32_t w, int32_t cs,
                            int32_t cw, int32_t cwide_buf, int32_t wide_coff, int32_t wide_is_out,
                            const float* mean, const float* std, b200_stream_t stream);

/* BatchNorm2d (training mode, batch statistics) + LeakyReLU on NHWC bf16 -- block.py:122,91.
 * b200_bn_stats_finalize: stats = fp32 [2][c] sum, sumsq over n*h*w (zeroed by the call); the block that produces
 * the totals also writes mean_invstd = [2][c] mean, invstd and updates the running statistics (when non-null) in
 * the same launch (nn.BatchNorm2d semantics).                                                                    */
int b200_bn_stats_finalize(const void* z, float* stats, float* mean_invstd, float* running_mean,
                           float* running_var, int64_t npix, int32_t c, float momentum, float eps,
                           b200_stream_t stream);
/* The finishing step of b200_bn_stats_finalize (stats -> mean_invstd + running statistics) for many layers in
 * one launch (the running-statistics side effect of a re-used train-mode forward: 11 layers x 2 re-used forwards
 * per step).  table: device array of b200_bn_finalize_entry.                                                    */
typedef struct {
  const float* stats;   /* [2][c] sum, sum of squares */
  float* mean_invstd;   /* [2][c] */
  float* running_mean;  /* [c] or NULL */
  float* running_var;   /* [c] or NULL */
  int64_t npix;
  int32_t c;
  float momentum, eps;
  int32_t pad_;
} b200_bn_finalize_entry;
int b200_bn_finalize_multi(const b200_bn_finalize_entry* table_dev, int32_t count, int32_t c_max,
                           b200_stream_t stream);
/* BatchNorm statistics from the conv epilogue instead of a pass over z: b200_conv_igemm_stats (below) writes one
 * row of per-channel (sum, sum of squares) per 128-pixel half tile into part[2][c][rows]; this adds the rows in a
 * fixed order and finishes like b200_bn_stats_finalize.  rows = b200_conv_igemm_stat_rows(desc).                */
int b200_bn_partials_finalize(const float* part, int32_t rows, float* stats, float* mean_invstd,
                              float* running_mean, float* running_var, int64_t npix, int32_t c, float momentum,
                              float eps, b200_stream_t stream);
int b200_bn_apply_lrelu(const void* z, const float* mean_invstd, const float* gamma,
                        const float* beta, void* a, int64_t npix, int32_t c, float slope,
                        b200_stream_t stream);
/* backward: da = grad wrt lrelu output.  Pass 1 reduces sums[2][c] = (sum dbn, sum dbn*zhat) deterministically and
 * accumulates dbeta += sums[0], dgamma += sums[1] when non-null; pass 2 writes dz.  use_batch_stats = 0 is the
 * eval()-mode backward (mean_invstd built from the running statistics: the batch-mean terms vanish).        */
int b200_bn_bwd_reduce(const void* z, const void* da, const float* mean_invstd,
                       const float* gamma, const float* beta, float* sums, float* dgamma, float* dbeta,
                       int64_t npix, int32_t c, float slope, b200_stream_t stream);
int b200_bn_bwd_apply(const void* z, const void* da, const float* mean_invstd, const float* gamma,
                      const float* beta, const float* sums, void* dz, int64_t npix, int32_t c, float slope,
                      int32_t use_batch_stats, b200_stream_t stream);

/* MaxPool2d(2,2) on NHWC bf16 (perceptual.py:158) and its backward fused with the ReLU mask
 * of the pooled activation.                                                                 */
int b200_maxpool2x2(const void* x, void* y, int32_t n, int32_t h, int32_t w, int32_t c,
                    b200_stream_t stream);
int b200_maxpool2x2_bwd(const void* x, const void* dy, void* dx, int32_t n, int32_t h, int32_t w,
                        int32_t c, b200_stream_t stream);

/* nearest x2 upsample backward: dx[n,y,x,c] = (sum of the 2x2 block of dy) * lrelu'(m) where m is
 * read from mask_up[n,2y,2x,c] (the upsampled activation itself, [n,2h,2w,c]) when non-null.   */
int b200_sumpool2x2_mask(const void* dy, const void* mask_up, void* dx, int32_t n, int32_t h,
                         int32_t w, int32_t c, float slope, b200_stream_t stream);
/* nn.PixelShuffle(2) on NHWC bf16 (+ LeakyReLU when act != 0), pixelshuffle_block block.py:374-387:
 * out[n, 2y+i, 2x+j, c'] = act(z[n, y, x, 4c' + 2i + j]);  z is [n,h,w,4c], out is [n,2h,2w,c].
 * b200_pixel_unshuffle2 is its transpose (the input gradient): dz[n,y,x,4c'+2i+j] = dout[n,2y+i,2x+j,c']. */
int b200_pixel_shuffle2(const void* z, void* out, int32_t n, int32_t h, int32_t w, int32_t c,
                        int32_t act, float slope, b200_stream_t stream);
int b200_pixel_unshuffle2(const void* dout, void* dz, int32_t n, int32_t h, int32_t w, int32_t c,
                          b200_stream_t stream);

/* L1 loss (mean |a-b|) forward + gradient in one pass -- losses.py:37-39.
 * fp32 variant: a, b fp32, grad_a fp32 = gscale*sign(a-b)/numel.  bf16 variant likewise.
 * loss_out: fp32 scalar accumulated with one atomic per block (zeroed by the call).        */
int b200_l1_loss_f32(const float* a, const float* b, float* loss_out, float* grad_a, int64_t numel,
                     float weight, b200_stream_t stream);
int b200_l1_loss_bf16(const void* a, const void* b, float* loss_out, void* grad_a, int64_t numel,
                      float weight, b200_stream_t stream);

/* elementwise helpers */
int b200_lrelu_mask_mul(const void* g, const void* y, void* out, int64_t numel, float slope,
                        b200_stream_t stream);
int b200_nchw_f32_to_nhwc_bf16(const float* x, void* y, int32_t n, int32_t c, int32_t h, int32_t w,
                               int32_t cy, int32_t y_coff, b200_stream_t stream);
int b200_nhwc_bf16_to_nchw_f32(const void* x, float* y, int32_t n, int32_t c, int32_t h, int32_t w,
                               int32_t cx, int32_t x_coff, b200_stream_t stream);

const char* b200_last_error(void);
int b200_version(void);
int b200_device_ok(void);   /* 1 if the current device is sm_100 */
int64_t b200_launch_count(void);  /* kernels launched by this library since load */

#ifdef __cplusplus
}
#endif
#endif /* TRAINNER_B200_H_ */
