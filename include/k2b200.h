/* k2b200.h -- C ABI of libk2b200.so, the B200 (sm_100a) kernel library behind the Kandinsky-2
 * denoising hot path.
 *
 * The reference (ai-forever/Kandinsky-2) has no FFI: its "operator API" for this path is the set of
 * PyTorch library calls issued by kandinsky2/model/unet.py, kandinsky2/model/nn.py,
 * kandinsky2/model/gaussian_diffusion.py and kandinsky2/vqgan/movq_modules.py.  Each entry point
 * below replaces one such call-site family (cited per function) and is what the Python boundary
 * modules in kandinsky-2_b200/kandinsky2/ bind through ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success and <0 on error; k2_last_error() gives the thread-local
 *     message; no C++ exception crosses the boundary;
 *   - all pointers are DEVICE pointers unless a parameter is documented as host memory; the library
 *     never allocates user-visible memory and never synchronises the device;
 *   - every launch is enqueued on the caller's stream (pass torch.cuda.current_stream().cuda_stream);
 *   - activations are NHWC fp16 ("rows" = pixels, row stride `ld*` in ELEMENTS so that a tensor may
 *     be a channel slice of a wider buffer); weights are pre-packed by the host (layout per function);
 *   - there is no CPU fallback: without an sm_100 device every call fails.
 */
#ifndef K2B200_H_
#define K2B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* k2_stream_t; /* cudaStream_t */

const char* k2_last_error(void);
int k2_version(void);
/* Number of kernels launched by this library in this process since the last reset (bench evidence). */
long long k2_launch_count(void);
void k2_reset_launch_count(void);
/* Tuning knobs: key 0 = force conv/GEMM N tile (0 = auto); key 1 = split-K (0 auto, 1 off, n>1 forced);
 * key 2 = CTA-pair kernel (0 auto, 1 off, 2 on); key 3 = halo 3x3 kernel (0 off, 1-4 layout variants);
 * key 4 = programmatic dependent launch (0/1); key 5 = cycles by which the attention kernel's second query tile starts late
 * (default 1200; each query tile has its own MMA-issuing thread, so the two tiles' softmax phases stay apart);
 * key 6 = attention softmax arithmetic: n = eighths (0..3) of the exponentials evaluated on the FMA pipe instead of MUFU,
 * + 10 = scale-and-subtract as packed FFMA2, + 30 = FFMA2 and packed FADD2 row sums (bit-identical to the same n), 200 = traced
 * (default 0); keys 7 / 8 = low / high 32 bits of a device buffer (384 x u64) that the traced attention variant fills with
 * clock64 stamps of CTA (0,0,0) -- diagnostics only, see profiles/attn_probe.py; key 9 = attention softmax layout (1 = 16 warps,
 * half a score row per thread, default; 0 = 8 warps, one row per thread);
 * key 10 = default number of epilogue warp sets of the CTA-pair conv kernel (1; 2 = 384-thread variant whose second set drains
 * the other half of the 64-column pairs: bit-identical results, faster where the K loop is short).  Keys 0, 1, 2 and 10 are
 * process-wide defaults; k2_conv_gemm_cfg overrides them per call.  key 11 = blocks per SM the GroupNorm apply grids are sized
 * for (0 = each kernel's real occupancy, i.e. one full wave; 4 = the round-1 sizing); key 12 = tail split of the CTA-pair conv
 * kernel's last partial wave (0 off, default; 1 = where the K loop is long enough to pay for the hand-over; 2 = wherever
 * possible: tests and probes). */
int k2_set_tuning(int key, int value);

/* ---------------------------------------------------------------------------------------------
 * Convolution / GEMM on tcgen05 tensor cores.
 * Replaces nn.Conv2d 3x3 (unet.py:152,180,426,562; movq_modules.py:139-148), nn.Conv2d 1x1
 * (unet.py:191; movq_modules.py:150-157,188-199) and nn.Conv1d k=1 (unet.py:251,257,258).
 *
 *   out[m, n] = bias[n] + residual[m, n] + sum_s sum_tap sum_c A_s[shift_tap(m), c] * Wp[n, k(s,tap,c)]
 *
 * m runs over the NB*H*W output pixels (NHWC order).  Up to 3 activation sources accumulate into the
 * same output; source s has `taps` = 9 (3x3, zero padding 1) or 1 (1x1).  Packed weights Wp are fp16
 * [w_rows >= Cout][Ktot], K contiguous, k ordered source-major, then tap (ky*3+kx), then channel, each
 * source's channel count padded to a multiple of 64 (zero weights for the padding).
 * out_mode 0: fp16 rows [M, ldo]; out_mode 1: fp32 NCHW [NB, Cout, H, W] (output heads).
 * ldw is the row stride of Wp in elements (0 = Ktot); a strided Wp lets an ACTIVATION matrix be the B operand
 * (MoVQ attention: scores = q k^T with k rows as "weights").
 * workspace (may be NULL): caller-owned scratch for split-K.  Where a cycle model of the launch (waves of work units x
 * K chunks per unit, plus the second pass) says so -- small M with a huge K -- K is split over several CTAs that write
 * fp32 partial tiles [split][M][Cout] there, and a second launch sums them in a fixed order (+bias, +residual) --
 * deterministic, no atomics.  The split-K partials use the LOWER half of the workspace.  The UPPER half serves the tail
 * split of the CTA-pair kernel (tuning key 12, off by default: measured neutral inside the power-capped step): when the last wave of work units would occupy only part of
 * the CTA pairs, each of its units is cut into 2..4 parts along K that run on the idle pairs, and the owning part adds the
 * others' fp32 accumulator tiles (handed over through the upper half, fixed summation order) before its ordinary epilogue --
 * one launch, same outputs and GroupNorm partials, a different (still deterministic) fp32 summation order.  The last
 * 64 KB of the workspace are hand-over flags: they must be ZERO before the first launch that uses the workspace; the library
 * leaves them zero after every launch.  Launches sharing a workspace must be stream-ordered.
 * gn_partial (may be NULL): fp32 [row groups][Cout][2]; when given and the launch qualifies (fp16 output, Cout % 64 == 0,
 * N tile >= 64) the launch also emits (sum, sum of squares) partials of the ROUNDED output, image-major, which
 * k2_gn_finalize turns into GroupNorm statistics -- the consumer's statistics pass disappears.  Row groups: one per M tile
 * when a tile lies inside one image; one per (image, spatial tile) for the (16 pixel x 8 image) tiles of tiny images; 16-row
 * groups from the second pass of a split-K launch.  gn_partial must hold max(M tiles*4, M/16)*Cout*2 floats
 * (k2_gn_scratch_floats); info[5] / info[6] tell what was written.
 * info (HOST pointer, may be NULL): int[7] = {N tile, CTA-pair mode, split-K factor, M tiles, images per tile,
 * gn_partial written (0 no / 1 epilogue / 2 split-K pass), row groups written in total}.
 * taps = 4 (allowed for a single source, fp16 output, no residual, H and W even): the source is [NB, H/2, W/2, C] and the call
 * computes the 3x3 convolution over its NEAREST-2x UPSAMPLING (unet.py:67-77 + :199-203; movq_modules.py:93-97) without
 * materialising it: output pixel (2y+a, 2x+b) = a 2x2 convolution of the source around (y, x) with the kernel rows / columns
 * that fall on the same source pixel pre-summed by the host (2.25x fewer MACs).  Wp = fp16 [Cout][16 * pad64(C)],
 * k = ((a*2+b)*4 + ty*2+tx) * pad64(C) + c, source offset (ty+a-1, tx+b-1); Ktot = 16 * pad64(C).
 * A plain GEMM [M,K]x[K,N] is the call with NB=1, H=1, W=M, one source with taps=1.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  const void* ptr; /* fp16, NHWC; may point at a channel offset inside a wider buffer */
  int C;           /* channels of this source (multiple of 8) */
  int ld;          /* row stride in elements */
  int taps;        /* 9, 1, or 4 (3x3 over the nearest-2x upsampled source, see above) */
} K2ConvSrc;

int k2_conv_gemm(const K2ConvSrc* srcs, int nsrc, int NB, int H, int W, const void* w_packed, int w_rows,
                 int Ktot, int ldw, int Cout, const float* bias, const void* residual, int ldr, void* out, int ldo,
                 int out_mode, void* workspace, long long workspace_bytes, float* gn_partial, int* info,
                 k2_stream_t stream);

/* k2_conv_gemm with the launch configuration chosen by the caller instead of the library's cycle model:
 * cfg (HOST pointer, may be NULL = k2_conv_gemm) = int[4] {N tile (16/64/128/192/256), CTA-pair kernel (1 off, 2 on),
 * split-K factor (1 = off), epilogue warp sets of the CTA-pair kernel (1 or 2)}; a 0 entry keeps the automatic choice.
 * N tile, pair mode and epilogue sets never change a result bit (same K order per output element); the split factor does.
 * The UNet / MoVQ launch plans time the candidates once per distinct layer shape and bake the winner into their CUDA graph.
 * w_batch_stride (elements, multiple of 8; 0 = one weight matrix): > 0 makes the call a BATCHED GEMM -- image n of the NB
 * images multiplies Wp + n * w_batch_stride.  This is how the MoVQ AttnBlock (movq_modules.py:201-225) runs without a loop
 * over images: scores[n] = q[n] k[n]^T with the k rows of image n as "weights" (w_rows = T, ldw = row stride of the qkv
 * buffer), out[n] = P[n] v[n] with v[n]^T as "weights".  Tiles then never span two images; no split-K. */
int k2_conv_gemm_cfg(const K2ConvSrc* srcs, int nsrc, int NB, int H, int W, const void* w_packed, int w_rows,
                     int Ktot, int ldw, int Cout, const float* bias, const void* residual, int ldr, void* out, int ldo,
                     int out_mode, void* workspace, long long workspace_bytes, float* gn_partial, int* info,
                     const int* cfg, long long w_batch_stride, k2_stream_t stream);

/* The decisions k2_conv_gemm takes for a geometry -- M tile box, N tile, CTA-pair mode, split-K factor, how the GroupNorm
 * partials come out -- without touching a pointer or the GPU (host arithmetic only; for tests, tooling and the caller's
 * scratch sizing).  taps: 9 if any source is a 3x3, else 1; Ktot as for k2_conv_gemm; workspace_bytes 0 = no workspace;
 * info = int[7] with the meaning given above. */
int k2_conv_plan(int NB, int H, int W, int taps, int Ktot, int Cout, int out_mode, long long workspace_bytes,
                 int want_gn_partial, int* info);

/* K parts the last partial wave's units were cut into (tail split, see k2_conv_gemm) by the most recent k2_conv_gemm /
 * k2_conv_gemm_cfg / k2_conv_plan call of this thread: 1 = not used.  Diagnostics for tests and tooling. */
int k2_conv_last_tail_split(void);

/* ---------------------------------------------------------------------------------------------
 * GroupNorm (32 groups in the UNet) statistics + fused apply.
 * Replaces GroupNorm32.forward (nn.py:31-37), the FiLM  norm(h)*(1+scale)+shift  and SiLU of
 * ResBlock.forward (unet.py:209-216), Upsample/Downsample on h and x (unet.py:67-77,105-107), the
 * torch.cat of the up path (text2im_model2_1.py:99) and MoVQ SpatialNorm (movq_modules.py:61-68).
 *
 * k2_gn_stats: per (image, group) mean and rstd of the channel-concatenation [src0 | src1]
 *   (src1 may be NULL); stats is fp32 [NB, groups, 2]; scratch is fp32 workspace of
 *   k2_gn_scratch_floats(NB, HW, C0+C1) floats that the caller ZEROES once at allocation (its first
 *   1024 words are self-resetting arrival counters); deterministic.
 * k2_gn_apply: y = act( ((x-mean)*rstd*gamma+beta) * (1+scale[n,c]) + shift[n,c] ), written as fp16
 *   rows of the concatenated tensor, optionally resampled:
 *     resample 0: same size; 1: 2x2 average pool of y (and of raw x into xres); 2: nearest 2x upsample.
 *   film is fp32 rows (scale[0..C) | shift[C..2C)) with row stride film_ld, or NULL.  act: 0 none, 1 SiLU.
 *   spatial (MoVQ): if zq != NULL, y = GN(x) * (Wy.zq + by) + (Wb.zq + bb) with zq fp32 NHWC
 *   [NB, zh, zw, 4] nearest-resized to (H, W); sn_w is fp32 [C, 10] = (Wy[4], by, Wb[4], bb).
 * ------------------------------------------------------------------------------------------- */
long long k2_gn_scratch_floats(int NB, int HW, int C);
int k2_gn_stats(const void* src0, int C0, int ld0, const void* src1, int C1, int ld1, int NB, int HW,
                int groups, float eps, float* stats, float* scratch, k2_stream_t stream);
/* statistics from the partials k2_conv_gemm wrote (one or two channel-concatenated sources of the same image size);
 * rg0 / rg1 = row groups per image of each source (info[6] / NB of the producing call). */
int k2_gn_finalize(const float* part0, int C0, int rg0, const float* part1, int C1, int rg1, int NB, int HW, int groups,
                   float eps, float* stats, k2_stream_t stream);
int k2_gn_apply(const void* src0, int C0, int ld0, const void* src1, int C1, int ld1, int NB, int H, int W,
                int groups, const float* stats, const float* gamma, const float* beta, const float* film,
                int film_ld, int act, int resample, void* y, int ldy, void* xres, int ldx, const float* zq, int zh,
                int zw, const float* sn_w, k2_stream_t stream);
/* k2_gn_apply with the statistics pass folded in: instead of `stats` the producers' partial sums (the part0 / rg0 / part1 / rg1
 * / eps arguments of k2_gn_finalize) are given and every block derives mean / rstd of the groups it touches itself -- one
 * launch less per GroupNorm.  No SpatialNorm inputs.  Statistics equal k2_gn_finalize's up to fp32 summation order
 * (tests/test_gpu_ops.py::test_gn_apply_fold_matches_finalize_plus_apply). */
int k2_gn_apply_fold(const void* src0, int C0, int ld0, const void* src1, int C1, int ld1, int NB, int H, int W, int groups,
                     const float* part0, int rg0, const float* part1, int rg1, float eps, const float* gamma,
                     const float* beta, const float* film, int film_ld, int act, int resample, void* y, int ldy, void* xres,
                     int ldx, k2_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Attention, head dim 64, online softmax, on tcgen05 (QK^T and PV) with encoder K/V prepended.
 * Replaces QKVAttention.forward (unet.py:286-340) incl. the optional flash-attn path (:303-332).
 *   qkv   fp16 [B, T, ldq] rows; head h owns channels [h*hs, (h+1)*hs) with q at +q_off, k at +k_off,
 *         v at +v_off (reference layout: hs=192, 0/64/128 -- unet.py:296).
 *   enc   fp16 [B, Tc, lde] rows or NULL (Tc=0); head h: k at h*ehs+ek_off, v at h*ehs+ev_off.
 *   out   fp16 [B, T, ldo], channel h*64+d.
 *   scale multiplies q.k (reference: 1/sqrt(64), applied as d^-1/4 on each operand, unet.py:334-337).
 * ------------------------------------------------------------------------------------------- */
int k2_attention_d64(const void* qkv, int ldq, int hs, int q_off, int k_off, int v_off, const void* enc,
                     int lde, int ehs, int ek_off, int ev_off, int B, int heads, int T, int Tc, float scale,
                     void* out, int ldo, k2_stream_t stream);

/* One head of width 512 over T tokens, no [T, T] score matrix: the MoVQ AttnBlock (movq_modules.py:201-225; the encoder's
 * twin vqgan_blocks.py:186-240).  qkv fp16 rows [B, T, ldq] with q / k / v at element offsets q_off / k_off / v_off (512 channels
 * each); out fp16 [B, T, ldo] (512 channels); scale multiplies q.k (the reference: C ** -0.5).  A CTA owns 128 queries and half
 * of the output channels (TMEM holds 256 columns of O + two score buffers), so the score tile is computed twice per query tile. */
int k2_attention_d512(const void* qkv, int ldq, int q_off, int k_off, int v_off, int B, int T, float scale, void* out, int ldo,
                      k2_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Small dense layers (fp32 math): nn.Linear (+ optional SiLU on the input and/or the output),
 * nn.LayerNorm, and the sinusoidal timestep embedding.
 * Replaces time_embed (unet.py:414-419), emb_layers (unet.py:166-172), the conditioning head
 * (text2im_model2_1.py:57-80) and timestep_embedding (nn.py:101-121).
 *   y[m, n] = (silu_out ? silu : id)( b[n] + sum_k (silu_in ? silu(x[m,k]) : x[m,k]) * W[n,k] ) (+ add[m,n])
 * x fp32 [M, K] (ldx), W fp16 or fp32 [N, K] (w_is_half), y fp32 [M, N] (ldy).
 * ------------------------------------------------------------------------------------------- */
int k2_linear(const float* x, int ldx, const void* W, int w_is_half, const float* b, const float* add,
              int ldadd, float* y, int ldy, int M, int N, int K, int silu_in, int silu_out,
              k2_stream_t stream);
int k2_layernorm(const float* x, const float* gamma, const float* beta, float* y, int M, int N, float eps,
                 k2_stream_t stream);
int k2_timestep_embedding(const float* t, float* out, int B, int dim, float max_period, k2_stream_t stream);
/* fp32 rows -> fp16 rows (context tokens), and generic strided copy helpers */
int k2_f32_to_f16(const float* x, void* y, long long n, k2_stream_t stream);
/* y = silu(x) on n fp16 elements, may run in place: the activations of the Kandinsky 2.2 ControlNet hint stem (diffusers
 * ImageHintTimeEmbedding.input_hint_block, once per generation; BASELINE configs[4]) */
int k2_silu_f16(const void* x, void* y, long long n, k2_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Stem im2col: fp32 NCHW latent (+ optional inpaint image*mask and mask, text2im_model2_1.py:146-155)
 * -> fp16 rows [NB*H*W, Kpad] holding the 3x3xCin patch (k = tap*Cin + c), zero padded, so that
 * input_blocks.0 (unet.py:426) runs through k2_conv_gemm as a GEMM.
 * ------------------------------------------------------------------------------------------- */
int k2_stem_im2col(const float* x, int Cx, const float* x2, int C2, const float* x3, int C3, int mul23,
                   int NB, int H, int W, void* out, int Kpad, k2_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Sampler step (classifier-free guidance + DDPM learned-range posterior), fused.
 * Replaces model_fn (kandinsky2_1_model.py:222-233), p_mean_variance / process_xstart / p_sample
 * (gaussian_diffusion.py:223-322,352-382) and denoised_fun (kandinsky2_1_model.py:237-243).
 *   model_out fp32 NCHW [2B, 8, H, W]; x fp32 [B, 4, H, W] (in place -> x_{t-1}); noise fp32 [B,4,H,W].
 *   coef (device, fp32[8]): sqrt_recip_ac, sqrt_recipm1_ac, post_coef1, post_coef2, min_log, max_log,
 *   nonzero, sqrt(alphas_cumprod[next timestep]) (2.2 inpainting only).  cond_first: 1 = rows [0,B) conditional (2.1), 0 = unconditional first (2.2).
 *   threshold_mode 0: x0 = clamp(x0, -clip, clip); 1: additionally the reference's dynamic threshold
 *   s = max(percentile_99.5(|x0[sample 0]|), 1); x0 = clip(x0, -s, s)/s   (gaussian_diffusion.py:284-294), the percentile
 *   bit-identical to np.percentile with numpy >= 2 semantics (float32 index, weight and interpolation).
 *   Split step for sharded runs (the reference's "sample 0" is GLOBAL sample 0): 2 = x0 + percentile of local sample 0 -> s in
 *   work[B*4*H*W], no update; 4 = x0 only; 3 = the update, with s read from work[B*4*H*W] (the caller broadcasts that float
 *   from the rank that owns global sample 0 between the two calls).
 *   Inpainting (mask fp32 [B,1,H,W], 1 = keep; init fp32 [B,4,H,W] = the clean latent):
 *     inpaint_noise == NULL (Kandinsky 2.1, kandinsky2_1_model.py:237-243): x0 = x0*(1-mask) + init*mask after the clamp;
 *     inpaint_noise != NULL (Kandinsky 2.2 = diffusers KandinskyV22InpaintPipeline, restated: not in /root/reference): x0 is
 *     left alone and  x_{t-1} = mask * (c*init + sqrt(1-c^2)*inpaint_noise) + (1-mask) * x_{t-1}  with c = coef[7] =
 *     sqrt(alphas_cumprod[next timestep]) (1 at the last step = the final blend with the clean latent); inpaint_noise fp32
 *     [B,4,H,W] is the run's initial latent noise.
 *   work: fp32 scratch of at least B*4*H*W + 4096 floats.
 * ------------------------------------------------------------------------------------------- */
int k2_sampler_step(const float* model_out, float* x, const float* noise, const float* coef, int B, int H,
                    int W, float guidance, int cond_first, float clip, int threshold_mode,
                    const float* inpaint_init, const float* inpaint_mask, const float* inpaint_noise, float* work,
                    k2_stream_t stream);

/* Device-side schedule of the sampling loop, so that a whole denoising step (latent duplication for CFG + UNet + guidance +
 * scheduler update) is one CUDA graph replayed once per step with nothing copied from the host (gaussian_diffusion.py:
 * 426-475 p_sample_loop_progressive runs the loop on the host).  `counter` is a device int[2] = (step, number of steps in the
 * schedule), written by the caller before step 0; with k = counter[0] % counter[1]:
 *   k2_step_begin: x_in[0:n) = x_in[n:2n) = x[0:n) (n = B*4*H*W);  t_in[0:nt) = ts_seq[k];  coef_out[0:8) = coef_seq[k][0:8);
 *                  noise[0:n) = noise_seq[k][0:n) if noise_seq != NULL (per-step noise drawn up front, one stream per image).
 *   k2_step_end:   counter[0] += 1. */
int k2_step_begin(const float* x, float* x_in, long long n, float* t_in, int nt, float* coef_out, const float* ts_seq,
                  const float* coef_seq, const float* noise_seq, float* noise, const int* counter, k2_stream_t stream);
int k2_step_end(int* counter, k2_stream_t stream);

/* PLMS / DDIM update with an explicit epsilon history (replaces PLMSSampler.p_sample_plms, samplers.py:571-637, and the
 * CFG closure): e_t = uncond + g (cond - uncond) from model_out's first 4 channels (C2 channels per sample);
 * e' = coef[4] e_t + coef[5] hist0 + coef[6] hist1 + coef[7] hist2 (NULL history entries are skipped);
 * out = coef[2] (coef[0] x - coef[1] e') + coef[3] e'; e_t is also written to `store` if not NULL.  coef is device fp32[8]
 * = {1/sqrt(a_t), sqrt(1-a_t)/sqrt(a_t), sqrt(a_prev), sqrt(1-a_prev), w0, w1, w2, w3}. */
int k2_plms_step(const float* model_out, int C2, const float* x, float* out, const float* hist0, const float* hist1,
                 const float* hist2, float* store, const float* coef, int B, int H, int W, float guidance, int cond_first,
                 k2_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * MoVQ helpers: nearest-codebook search (quntize.py:89-98; fp32, ties -> lowest index, int64 out),
 * fp32 NCHW -> NHWC transposes for the 4-channel latent, final image quantisation
 * (utils.py:57-70: ((x+1)*127.5).round().clamp(0,255) -> uint8 NHWC).
 * ------------------------------------------------------------------------------------------- */
int k2_vq_argmin(const float* z, const float* codebook, long long* idx, int n, int n_embed, int dim,
                 k2_stream_t stream);
/* y[n,o,:] = b[o] + sum_i w[o,i] x[n,i,:] on fp32 NCHW (MoVQ post_quant_conv 4->4, autoencoder.py:183) */
int k2_pointwise_nchw_f32(const float* x, const float* w, const float* b, float* y, int NB, int Ci, int Co, int HW,
                          k2_stream_t stream);
/* nearest 2x upsample of fp16 NHWC rows (movq_modules.py:93-97 F.interpolate before the conv) */
int k2_upsample2x_nhwc(const void* x, int ldx, void* y, int ldy, int NB, int H, int W, int C, k2_stream_t stream);
/* y[n, yo, xo, :] = x[n, 2*yo+oy, 2*xo+ox, :] on fp16 NHWC rows.  With (oy, ox) = (1, 1) applied to a stride-1 'same' 3x3
 * conv this is the VQGAN encoder's Downsample: pad (0,1,0,1) + conv3x3 stride 2 (vqgan_blocks.py:109-126). */
int k2_subsample2_nhwc(const void* x, int ldx, void* y, int ldy, int NB, int H, int W, int C, int oy, int ox,
                       k2_stream_t stream);
/* y[r, :] = softmax(scale * x[r, :]) over n columns, fp16 in/out, fp32 math (movq_modules.py:213-215) */
int k2_softmax_rows(const void* x, int ldx, void* y, int ldy, long long rows, int n, float scale, k2_stream_t stream);
int k2_nchw_to_nhwc_f32(const float* x, float* y, int NB, int C, int H, int W, k2_stream_t stream);
int k2_images_to_u8(const float* x_nchw, uint8_t* out_nhwc, int NB, int C, int H, int W, int crop_h,
                    int crop_w, k2_stream_t stream);
/* MoVQ SpatialNorm (movq_modules.py:61-68) + optional swish (:21-23), one read + one write of the feature map:
 *   y = act( GroupNorm(x) * (Wy.zq + by) + (Wb.zq + bb) ),  zq fp32 NHWC [NB, zh, zw, 4] nearest-resized to (H, W),
 * stats fp32 [NB, groups, 2] (mean, rstd) from k2_gn_finalize / k2_gn_stats, sn_w fp32 [C, 10] = (Wy[4], by, Wb[4], bb).
 * The per-channel normalisation and both 4 -> C modulations are folded into 10 register-resident coefficients per channel. */
int k2_sn_apply(const void* x, int C, int ldx, int NB, int H, int W, int groups, const float* stats, const float* gamma,
                const float* beta, const float* zq, int zh, int zw, const float* sn_w, int act, void* y, int ldy,
                k2_stream_t stream);
/* fp16 rows [B][T][ldx] (C columns) -> [B][C][T] (the attention values as a K-major B operand, movq_modules.py:216-219) */
int k2_transpose_f16(const void* x, int ldx, void* y, int B, int T, int C, k2_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Diffusion prior (SURVEY.md 8f rank 3; kandinsky2/model/prior.py:46-127), not on the measured denoising path and not
 * tuned.  The transformer's Linear layers are k2_conv_gemm flat-row GEMMs; these are the rest:
 *   k2_layernorm_f16   LayerNorm over the last dim of fp16 rows, fp32 statistics / gain / bias (prior.py:46-53)
 *   k2_gelu_f16        nn.GELU (exact erf) on n fp16 elements, may run in place (prior.py:74-83)
 *   k2_attention_small QKVMultiheadAttention for T <= 128 tokens, head dim 64 (prior.py:86-103): qkv rows
 *                      [B, T, >= heads*192] with per-head [q | k | v]; additive mask = causal (if set) AND key keep-mask
 *                      (uint8 [B, T], may be NULL); fp32 softmax; out rows [B, T, >= heads*64].
 * ------------------------------------------------------------------------------------------- */
int k2_layernorm_f16(const void* x, int ldx, const float* gamma, const float* beta, void* y, int ldy, int M, int N, float eps,
                     k2_stream_t stream);
int k2_gelu_f16(const void* x, void* y, long long n, k2_stream_t stream);
int k2_attention_small(const void* qkv, int ldq, const unsigned char* keep_mask, int causal, void* out, int ldo, int B, int T,
                       int heads, float scale, k2_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* K2B200_H_ */
