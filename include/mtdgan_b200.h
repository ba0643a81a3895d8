/* libmtdgan_sm100a.so — C ABI of the B200-native MTD-GAN hot path.
 *
 * The reference (babbu3682/MTD-GAN) is pure Python/PyTorch and has no FFI of its own; the interface
 * each entry point replaces is therefore the PyTorch call the reference makes at the cited
 * file:line (all under /root/reference).  INTEGRATION.md shows the ctypes binding a maintainer adds.
 *
 * Conventions (SURVEY §8b)
 *  - Plain pointers and sizes only; every pointer is a DEVICE pointer to fp32 data unless stated.
 *  - Activations are NHWC contiguous: (B, H, W, C).  The reference's NCHW tensors have C == 1 at the
 *    module boundaries (images, decision maps), where both layouts coincide; mtd_layout_transpose
 *    converts where a multi-channel module is called stand-alone.
 *  - The caller owns all memory, including workspaces; nothing is allocated or freed here.
 *  - All work is enqueued on `stream` (a cudaStream_t passed as void*); no implicit synchronisation;
 *    graph-capturable.  Stateless and re-entrant.
 *  - Return value: 0 ok; < 0 argument / shape error (MTD_EINVAL -1, MTD_EALIGN -2); > 0 a cudaError_t.
 *  - There is NO CPU implementation behind any entry point.
 */
#ifndef MTDGAN_B200_H_
#define MTDGAN_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

/* activation codes */
#define MTD_ACT_NONE_C 0
#define MTD_ACT_RELU_C 1
#define MTD_ACT_LEAKY_C 2

/* ---- library info ---------------------------------------------------------------------------- */
int mtd_abi_version(void);
/* 1 if the running device is compute capability 10.x (B200), else 0; <0 on CUDA error */
int mtd_device_ok(void);
/* number of CUDA kernels this library has launched in this process (host-side counter) */
long long mtd_kernel_launch_count(void);
/* programmatic dependent launch (every kernel waits on griddepcontrol before touching memory and lets the next
 * grid be scheduled early); on by default, returns the previous setting.  Off = plain stream serialization.   */
int mtd_set_pdl(int enabled);

/* ---- convolution (conv_simt.cu, conv_tc.cu) ----------------------------------------------------
 * Replaces nn.Conv2d / nn.ConvTranspose2d / nn.Linear forward and ATen convolution_backward:
 * arch/Ours/networks.py:18-19 (FFT_ConvBlock convs), :41-46 (generator encoder/decoder), :170
 * (UpsampleBlock), :181-306 (discriminator), applied at :32, :97-162, :385-472.
 *
 * Packed weight layouts (K-major for NHWC implicit GEMM):
 *   forward : wp[Cout][kh*kw][Cin]
 *   dgrad   : stride 1: wpd[Cin][kh*kw][Cout]; stride 2 (4x4, pad 1): wpd[4][Cin][4][Cout]
 * `transposed` = 1 for a ConvTranspose2d(stride 1) weight (Cin, Cout, kh, kw)  (SURVEY A6).      */
int mtd_conv_pack_fwd(const float* w_ref, int transposed, int Cout, int Cin, int kh, int kw, float* out, void* stream);
int mtd_conv_pack_dgrad(const float* w_ref, int transposed, int Cout, int Cin, int kh, int kw, int stride, float* out,
                        void* stream);
/* the same packs in the tile-major layout the tcgen05 kernels consume: [rows/32][K/32][32][32], K = kh*kw*channels
 * (every 32x32 tile is 4 KB contiguous, so a TMA weight box is a few contiguous runs), TF32 operand preparation
 * fused in: tf32 = 0 fp32 copy, 1 rounded to nearest tf32, 3 [hi | lo] split for the 3xTF32 mode (out: 2 x numel).
 * Needs Cout, Cin % 32 == 0. */
int mtd_conv_pack_fwd_blocked(const float* w_ref, int transposed, int Cout, int Cin, int kh, int kw, int tf32, float* out,
                              void* stream);
int mtd_conv_pack_dgrad_blocked(const float* w_ref, int transposed, int Cout, int Cin, int kh, int kw, int stride, int tf32,
                                float* out, void* stream);
/* Batched packing: between _begin and _end every pack entry point above records its work instead of launching; _end
 * launches it all, 24 packs per kernel (descriptions travel in kernel-parameter space: no table upload, graph-safe).
 * Host-side recording state: one batch at a time, not thread-safe.                                          */
int mtd_conv_pack_batch_begin(void);
int mtd_conv_pack_batch_end(void* stream);
/* y = post_act( pre_act( scale * conv(cat[x1,x2]) + bias ) + add1 + add2 );  aux (optional) receives the
 * value after pre_act.  x2/C2 = second source concatenated along channels (torch.cat at
 * networks.py:421-466) or null/0.  scale = device scalar 1/sigma of spectral norm, or null.  scale_group > 0 (all four
 * conv entry points): the batch holds several independent reference calls of scale_group samples each (e.g. D(real)
 * and D(fake) evaluated as one batch), every group with its own power-iteration result: scale is then an array with
 * one 1/sigma per group, applied by sample index / scale_group.  0 = one scalar.                              */
int mtd_conv_fwd(const float* x1, const float* x2, const float* wp, const float* bias, const float* scale, int scale_group,
                 float* y,
                 float* aux, const float* add1, const float* add2, int B, int H, int W, int C1, int C2, int N, int kh,
                 int kw, int stride, int pad, int pre_act, int post_act, float slope, void* stream);
/* dx = (scale * dgrad(dz) + add1 + add2) * act'(mask_src);  (H, W) are the conv INPUT dims.        */
int mtd_conv_dgrad(const float* dz, const float* wpd, float* dx, const float* scale, int scale_group, const float* add1,
                   const float* add2, const float* mask_src, int mask_act, float slope, int B, int H, int W, int Cin,
                   int Cout, int kh, int kw, int stride, int pad, void* stream);
/* gp[N][kh*kw][C1+C2] = sum over output pixels of dz (x) x   (dL/dW~ in packed forward layout)      */
int mtd_conv_wgrad(const float* x1, const float* x2, const float* dz, float* gp, int B, int H, int W, int C1, int C2,
                   int N, int kh, int kw, int stride, int pad, void* stream);
/* packed gradient -> reference layout; with inv_sigma != null applies the spectral-norm backward
 * dW_orig = (G - <G,W~> u v^T)/sigma (torch.nn.utils.spectral_norm; SURVEY A5).  scratch: 16 bytes.  */
int mtd_conv_wgrad_finish(const float* gp, float* dw_ref, int transposed, int Cout, int Cin, int kh, int kw,
                          const float* w_ref, const float* u, const float* v, const float* inv_sigma, void* scratch,
                          void* stream);
/* batched mtd_conv_wgrad_finish for every (layer, forward instance) of one backward pass; contributions of the
 * instances that share a weight are summed into one dw.  Segment table int64[n][16] = { gp, dw, w_ref, u, v,
 * inv_sigma, Cout, kh*kw, Cin, sN, sC, flip, sn_cols, dot slot, next segment of the same weight or -1,
 * pointer to a precomputed <G,W~> (mtd_act_bwd_sn) or 0 }
 * (Conv2d: sN = Cin*T, sC = T, flip 0; ConvTranspose2d: sN = T, sC = Cout*T, flip 1; flip bits 2 / 4: see
 * mtd_act_bwd_sn).  dot_chunks lists every
 * spectral-normed segment, head_chunks only the first segment of each weight.                              */
/* mtd_act_bwd for spectrally-normalised layers: also accumulates zw[g] += sum over the rows of batched call g of
 * dz . (y_pre - bias) = <G_g, W_orig>/sigma_g, the coefficient of the spectral-norm weight-gradient correction
 * (replaces the dot pass of the finishing step: segment field 15 = pointer to zw[g]).  dbias and zw pre-zeroed;
 * act = none or leaky.  dz_scale (optional, one 1/sigma per call): the dz written is pre-scaled, so dgrad needs no
 * scale and one weight-gradient GEMM over the whole batch gives sum_g G_g/sigma_g (segment flag bits: 2 = gp is
 * pre-scaled, 4 = correction-only instance without a gp).                                                  */
int mtd_act_bwd_sn(const float* dy, const float* y, float* dz, float* dbias, const float* bias, double* zw,
                   const float* dz_scale, int groups, long long M, int N, int act, float slope, void* stream);
/* mtd_act_bwd of one backward pass that also folds its dz into accumulators spanning several passes over the same
 * forward graph (the gradient of a sum of losses is linear in dz): dz (optional, unscaled, as mtd_act_bwd writes it);
 * acc[M][N] = (acc_first ? 0 : acc) + dz * inv_sigma[g] (inv_sigma optional: scale 1); dbias (optional) += column sums
 * of dz; zw (optional, as mtd_act_bwd_sn: act none or leaky) += per-call sums of dz . (y_pre - bias).  The batch
 * holds `groups` (<= 4) calls of M/groups rows.  y may be null when act is none and zw is null.  dbias and zw are
 * accumulated (zero them before the first pass).  Any N <= 8192.                                             */
int mtd_act_bwd_acc(const float* dy, const float* y, float* dz, float* acc, int acc_first, float* dbias, const float* bias,
                    double* zw, const float* inv_sigma, int groups, long long M, int N, int act, float slope, void* stream);
/* elements per chunk-table entry of a segment with kh*kw = taps and Cin = cin: a whole number of packed rows when a
 * row fits the kernels' shared-memory staging (coalesced transposition), else a fixed block                     */
int mtd_wgrad_finish_chunk_elems(int taps, int cin);
int mtd_wgrad_finish_batched(const void* seg_tab, int n_segs, const void* dot_chunks, int n_dot_chunks, const void* head_chunks,
                             int n_head_chunks, double* dots, void* stream);
/* dz = dy * act'(y) (F.relu / nn.LeakyReLU(0.2) backward); dbias[N] = column sums of dz (optional)  */
int mtd_act_bwd(const float* dy, const float* y, float* dz, float* dbias, int dbias_zeroed, long long M, int N, int act, float slope,
                void* stream);

/* tcgen05 / TMEM TF32 implicit-GEMM forward for C % 32 == 0 layers (conv_tc.cu).  Same contract as
 * mtd_conv_fwd restricted to one or two sources with C1 % 32 == 0 && C2 % 32 == 0, N % 32 == 0,
 * stride 1, power-of-two spatial dims; skinny-M layers are split-K; returns MTD_EINVAL for anything else (the caller then
 * uses mtd_conv_fwd).  passes = 1: TF32 operands, fp32 accumulate (rel. error <= 2e-3), wp tf32-rounded;
 * passes = 3: error-compensated 3xTF32 (fp32-grade, <= 1e-5), wp = [hi | lo] from mtd_split_tf32.  */
int mtd_conv_fwd_tc_supported(int B, int H, int W, int C1, int C2, int N, int kh, int kw, int stride, int pad);
/* kernel generation of the forward/dgrad tensor-core path: 1 = A through shared memory, 2 = A through TMEM with
 * several pixel tiles per CTA (weights streamed once per group).  Returns the previous setting.              */
int mtd_tc_set_version(int version);
/* tuning hook: force the Cout tile width (32/64/128) and/or the stream-K piece length (k-steps per CTA, -1 = whole
 * tiles only) of the forward/dgrad tensor-core kernel; 0 = chosen by the built-in cost model (the default).     */
int mtd_tc_set_tuning(int bn, int sk_per);
int mtd_tc_set_c32(int enabled);   /* 1 (default): 32->32 3x3 layers on the halo-tile kernel; returns the previous value */
int mtd_tc_set_halo(int enabled);  /* 1 (default): 3x3 stride-1 layers with > 32 channels on the streamed-weight halo-tile kernel; returns the previous value */
/* in-place round-to-nearest fp32 -> tf32 of a packed weight buffer (tcgen05 truncates its operands)  */
int mtd_round_tf32(float* p, long long n, void* stream);
/* ws / ws_floats (both TC entry points): caller-owned fp32 scratch (contents undefined before and after; one per
 * stream).  With it, layers whose tile count is not a multiple of the SM count run their remainder as a stream-K wave
 * (k-range pieces -> partial tiles in ws -> ordered reduction + epilogue): balanced SMs, deterministic, no atomics.
 * ws = NULL: whole output tiles only (correct, slower for skinny layers).  32 MB covers every layer of the model. */
int mtd_conv_fwd_tc(const float* x1, const float* x2, const float* wp, const float* bias, const float* scale, int scale_group,
                    float* y,
                    float* aux, const float* add1, const float* add2, int B, int H, int W, int C1, int C2, int N, int kh,
                    int kw, int stride, int pad, int pre_act, int post_act, float slope, int passes, float* ws, long long ws_floats,
                    void* stream);
/* dgrad on the tensor cores (stride 1, or stride 2 with 4x4/pad 1); same contract as mtd_conv_dgrad.
 * passes = 1: wpd tf32-rounded (mtd_round_tf32); passes = 3: wpd = [hi | lo] halves of the full dgrad pack
 * (mtd_split_tf32); for stride 1 wpd may point at a row slice of the hi half of [cin_total][T][Cout].
 * dx2 / c_split (stride 1, optional): the layer's input was torch.cat of two tensors -- input channels [0, c_split)
 * are written to dx (B,H,W,c_split) and the rest to dx2 (B,H,W,Cin-c_split) by ONE launch (dz is streamed once).  */
int mtd_conv_dgrad_tc(const float* dz, const float* wpd, float* dx, const float* scale, int scale_group, const float* add1,
                      const float* add2,
                      const float* mask_src, int mask_act, float slope, int B, int H, int W, int Cin, int Cout, int kh, int kw,
                      int stride, int pad, int passes, int cin_total, float* dx2, int c_split, float* ws, long long ws_floats,
                      void* stream);
/* weight gradient on the tensor cores (stride-1 same convs, C % 32 == 0, N % 32 == 0): both operands are
 * MN-major TMA boxes, split-K over pixels, fp32 atomics into gp (zeroed here).  Same gp layout as
 * mtd_conv_wgrad.                                                                                    */
int mtd_conv_wgrad_tc_supported(int B, int H, int W, int C1, int C2, int N, int kh, int kw, int stride, int pad);
int mtd_conv_wgrad_tc(const float* x1, const float* x2, const float* dz, float* gp, int B, int H, int W, int C1, int C2, int N,
                      int kh, int kw, int stride, int pad, int passes, void* stream);
/* the plan mtd_conv_wgrad_tc runs for these arguments: plan[5] = {1 halo kernel / 0 tap-streaming kernel, Cout tile,
 * split over pixels, pixel tiles per piece, CTAs}                                                        */
int mtd_conv_wgrad_tc_plan(int B, int H, int W, int C1, int C2, int N, int kh, int kw, int stride, int pad, int passes,
                           int* plan);
/* in place hi <- rna_tf32(w), lo <- rna_tf32(w - hi): operand split for the 3xTF32 mode               */
int mtd_split_tf32(float* hi, float* lo, long long n, void* stream);

/* ---- Res-FFT-Conv frequency branch (fft_block.cu) ------------------------------------------------
 * Replaces torch.fft.rfft2 / cat / fft_conv 1x1 + ReLU / chunk / complex / torch.fft.irfft2 at
 * arch/Ours/networks.py:24-29 and their autograd backward.  Half spectrum layout:
 * spec[B][W/2+1][H][C] complex64 (interleaved); C == 32 for the mix.                              */
/* 1 when the frequency branch supports the geometry: C == 32 and 1 <= H, W <= 512.  Lengths 64, 128, 256, 512 run four-step
 * FFTs (8x8 ... 16x32); every other length a Bluestein transform on a power-of-two length up to 1024.  The backward
 * (mtd_fft_cols_mix_bwd) takes H in {64, 128, 256} and W in {64, 128, 256, 512} only. */
int mtd_fft_supported(int H, int W, int C);
long long mtd_fft_spec_elems(int B, int H, int W, int C);          /* floats in a spectrum buffer      */
long long mtd_fft_bwd_part_elems(int B, int W);                    /* floats in the bwd partial buffer */
int mtd_fft_rows_fwd(const float* x, float* spec, int B, int H, int W, int C, void* stream);
int mtd_fft_cols_mix(const float* spec_in, float* spec_out, const float* w, const float* bias, int B, int H, int W,
                     int C, void* stream);
/* out = irfft-rows(spec) + add1 + add2  (the block's `x + img + fft`, networks.py:35)             */
int mtd_fft_rows_inv(const float* spec, const float* add1, const float* add2, float* out, int B, int H, int W, int C,
                     void* stream);
int mtd_fft_cols_mix_bwd(const float* spec_x, const float* spec_g, float* spec_out, const float* w, const float* bias,
                         float* part, float* dw, float* db, int B, int H, int W, int C, void* stream);

/* ---- spectral norm (spectral_norm.cu) ------------------------------------------------------------
 * Replaces the forward-pre-hook of nn.utils.spectral_norm (networks.py:181-300) for all layers of a
 * discriminator forward at once.  Tables are device arrays built by the host mirror: layer table
 * int64[L][8] = { W, u, v, rows, cols, u_off, v_off, p_off }; t_ws holds the per-row-block partial sums of W^T u
 * (sum over layers of ceil(rows / mtd_sn_rows_per_wtu_item()) * cols floats, p_off = the layer's slice), reduced
 * in a fixed order: u, v, sigma are bit-reproducible and identical on every data-parallel rank.     */
int mtd_sn_rows_per_wtu_item(void);
int mtd_sn_power_iter(const void* layer_tab, int n_layers, const void* work_wtu, int n_wtu, const void* work_wv,
                      int n_wv, float* t_ws, long long t_elems, float* s_ws, float* u_snap, float* v_snap,
                      float* inv_sigma, int update, float eps, void* stream);

/* ---- resampling / elementwise (resample.cu) -------------------------------------------------------
 * nn.Upsample(x2, bilinear) networks.py:230-260; nn.PixelShuffle(2) :171; .clip(0,1) :1969-1970;
 * nn.Dropout mask multiply :417.                                                                  */
int mtd_upsample2x_fwd(const float* in, float* out, int B, int H, int W, int C, void* stream);
int mtd_upsample2x_bwd(const float* dout, float* din, int B, int H, int W, int C, void* stream);
int mtd_pixel_shuffle2(const float* in, float* out, int B, int H, int W, int C, int backward, void* stream);
int mtd_layout_transpose(const float* in, float* out, int B, int C, int HW, int to_nhwc, void* stream);
int mtd_clip01_fwd(const float* x, float* y, long long n, void* stream);
int mtd_clip01_bwd(const float* x, const float* dy, float* dx, long long n, void* stream);
int mtd_mul(const float* a, const float* b, float* out, long long n, void* stream);
int mtd_add3(const float* a, const float* b, const float* c, float* out, long long n, void* stream);

/* ---- losses (losses.cu) ----------------------------------------------------------------------------
 * ls_gan losses.py:10-11; NDS_Loss :13-15; F.l1_loss / F.mse_loss networks.py:1964-1975;
 * CharbonnierLoss losses.py:108-111; EdgeLoss :122-138.  `acc` are fp64 device accumulators.       */
int mtd_nds_mask(const float* x, const float* y, unsigned char* mask, long long n, void* stream);
int mtd_sum_sqerr(const float* in, float target, const float* x, const float* y, long long n, double* acc, void* stream);
int mtd_sqerr_bwd(const float* in, float target, const float* x, const float* y, long long n, const float* gout, int k,
                  float scale, float* din, void* stream);
int mtd_sum_diff(const float* a, const float* b, long long n, int mode, float eps, double* acc, void* stream);
int mtd_diff_bwd(const float* a, const float* b, long long n, int mode, float eps, const float* gout, int k, float scale,
                 float* da, float* db, void* stream);
int mtd_sum_edge(const float* x, const float* y, int B, int H, int W, float eps, double* acc, void* stream);
int mtd_edge_bwd(const float* x, const float* y, int B, int H, int W, float eps, const float* gout, int k_edge,
                 float scale_edge, int k_pix, float scale_pix, float* dx, void* stream);
int mtd_loss_finalize(const double* acc, int k, float s0, float s1, float s2, float s3, float* out, void* stream);

/* ---- PCGrad (pcgrad.cu) -----------------------------------------------------------------------------
 * Replaces PCGrad._project_conflicting of module/weight_methods.py:449-464 and module/pcgrad.py:50-70. */
int mtd_pcgrad_chunk_elems(void);
/* out_seg = scale_seg * g_0 for every segment (same tables): gathers gradient tensors into one flat collective operand */
int mtd_segments_scale_copy(const void* seg_tab, const void* chunk_tab, int n_chunks, void* stream);
int mtd_pcgrad_gram(const void* seg_tab, const void* chunk_tab, int n_chunks, int T, double* gram_ws, void* stream);
int mtd_pcgrad_solve_combine(const void* seg_tab, const void* chunk_tab, int n_chunks, int T, const int* orders, int mean,
                             double* gram_ws, float* coef_out, float* cmat_out, double* gram_out, void* stream);
int mtd_pcgrad_project(const void* seg_tab, const void* chunk_tab, int n_chunks, int T, const int* orders, int mean,
                       double* gram_ws, float* coef_out, float* cmat_out, double* gram_out, void* stream);

/* ---- AdamW (adamw.cu) — "next" row: torch.optim.AdamW step of optimizers.py:9 / engine.py:44,52 ------
 * seg table int64[nseg][8]: { param, grad, exp_avg, exp_avg_sq, numel, step counter (device float*), 0, 0 };
 * the step counters are incremented on the device, bias corrections derived in-kernel (graph-capturable).
 * chunk table as PCGrad.
 * lr_dev (optional device float*): when non-NULL the learning rate is read from it instead of `lr`, so a captured
 * CUDA graph follows an lr scheduler.  grad_scale multiplies every gradient on the fly (1/world_size of a summed
 * all-reduce).  Bias corrections are evaluated in double like torch.optim.AdamW.                       */
int mtd_adamw_step(const void* seg_tab, int n_segs, const void* chunk_tab, int n_chunks, float lr, const float* lr_dev,
                   float beta1, float beta2, float eps, float weight_decay, float grad_scale, void* stream);

/* ---- data edge (data_edge.cu) — "next" row: the `window_patch` / `window` transform chains of
 * create_datasets/Mayo.py:117-136, 158-167 on int16 HU slices resident in HBM.
 * mtd_hu_foreground_bbox: bbox int32[S][4] = {y0, y1, x0, x1} (half-open) of {hu > a_min} per slice (CropForegroundd with
 *   select_fn x > 0 after windowing), {0,0,0,0} for an empty slice.
 * mtd_window_crop_patches: patch table int32[n][8] = {slice, oy, ox, by0, by1, bx0, bx1, aug} — (oy, ox) = slice
 *   coordinates of crop pixel (0,0) (negative inside SpatialPadd padding), [by0,by1) x [bx0,bx1) the foreground box (pixels
 *   outside it are padding zeros), aug bits 0-1 = RandRotate90d k, bit 2 = RandFlipd over both axes; writes the windowed
 *   low-dose / full-dose patches x, y (n, roi, roi) float32.
 * mtd_window_slices: ScaleIntensityRanged(a_min, a_max, 0, 1, clip=True) of whole slices (valid / test transform).  */
int mtd_hu_foreground_bbox(const short* hu, int S, int H, int W, float a_min, int* bbox, void* stream);
int mtd_window_crop_patches(const short* lo, const short* hi, int S, int H, int W, const int* patch_tab, int n_patches, int roi,
                            float a_min, float a_max, float* x, float* y, void* stream);
int mtd_window_slices(const short* hu, long long n, float a_min, float a_max, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MTDGAN_B200_H_ */
