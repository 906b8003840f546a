// k2_misc.cu -- the small kernels of the path: dense layers on tiny M, LayerNorm, timestep embedding,
// stem im2col, the fused classifier-free-guidance + DDPM sampler step, and the MoVQ helpers.
// Reference call sites are cited at each entry point (declared in include/k2b200.h).
#include <math.h>

#include "../../include/k2b200.h"
#include "k2_common.cuh"
#include "k2_internal.h"

namespace k2 {
namespace {

// ------------------------------------------------------------------------------------------------
// linear: one warp per output column, MT rows of x per pass. Weight rows are streamed once per row tile
// with 16-byte loads (fp16) -- this is a bandwidth-bound GEMV-like op (M = 2*batch rows).
// ------------------------------------------------------------------------------------------------
constexpr int LIN_MT = 8;   // rows of x staged in shared memory per block
constexpr int LIN_CB = 4;   // output columns per warp pass (register blocking over the staged x)
constexpr int LIN_NI = 4;   // column groups per warp (amortises the staging of x)

template <bool W_HALF>
__global__ void __launch_bounds__(256) linear_kernel(const float* __restrict__ x, int ldx, const void* __restrict__ Wv,
                                                     const float* __restrict__ b, const float* __restrict__ add,
                                                     int ldadd, float* __restrict__ y, int ldy, int M, int N, int K,
                                                     int Kp, int vec_ok, int silu_in, int silu_out, int ni) {
  extern __shared__ float xs[];  // [LIN_MT][Kp]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_wait();
  pdl_launch();
  const int m0 = blockIdx.y * LIN_MT;
  const int mt = min(LIN_MT, M - m0);
  for (int idx = threadIdx.x; idx < LIN_MT * Kp; idx += blockDim.x) {
    const int r = idx / Kp, k = idx - r * Kp;
    float v = 0.f;
    if (r < mt && k < K) {
      v = x[static_cast<long long>(m0 + r) * ldx + k];
      if (silu_in) v = silu_f(v);
    }
    xs[idx] = v;
  }
  __syncthreads();
  // each warp walks LIN_NI groups of LIN_CB output columns, so one staging of x serves 8 * LIN_CB * LIN_NI columns
  for (int it = 0; it < ni; ++it) {
    const int n0 = ((blockIdx.x * ni + it) * 8 + warp) * LIN_CB;
    if (n0 >= N) break;
    float acc[LIN_CB][LIN_MT];
#pragma unroll
    for (int cb = 0; cb < LIN_CB; ++cb)
#pragma unroll
      for (int i = 0; i < LIN_MT; ++i) acc[cb][i] = 0.f;
    const int K8 = vec_ok ? (K & ~7) : 0;
    // weights are streamed once from HBM: the raw 16-byte pieces of the NEXT k step are requested before the FMAs of the
    // current one (one warp would otherwise expose a full memory round trip per step)
    constexpr int RW = W_HALF ? 1 : 2;
    uint4 raw[LIN_CB][RW], nxt[LIN_CB][RW];
    auto fetch = [&](int k, uint4 (&dst)[LIN_CB][RW]) {
#pragma unroll
      for (int cb = 0; cb < LIN_CB; ++cb) {
#pragma unroll
        for (int q = 0; q < RW; ++q) dst[cb][q] = make_uint4(0u, 0u, 0u, 0u);
        if (n0 + cb < N) {
          const long long off = static_cast<long long>(n0 + cb) * K + k;
          if (W_HALF) {
            dst[cb][0] = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(Wv) + off));
          } else {
            const uint4* wp = reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(Wv) + off);
            dst[cb][0] = __ldg(wp);
            dst[cb][RW - 1] = __ldg(wp + (RW - 1));
          }
        }
      }
    };
    if (lane * 8 < K8) fetch(lane * 8, raw);
#pragma unroll 2
    for (int k = lane * 8; k < K8; k += 256) {
      if (k + 256 < K8) fetch(k + 256, nxt);
      float w[LIN_CB][8];
#pragma unroll
      for (int cb = 0; cb < LIN_CB; ++cb) {
        if (W_HALF) {
          const __half2* h2 = reinterpret_cast<const __half2*>(&raw[cb][0]);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 t = __half22float2(h2[e]);
            w[cb][2 * e] = t.x;
            w[cb][2 * e + 1] = t.y;
          }
        } else {
          const float* f = reinterpret_cast<const float*>(&raw[cb][0]);
#pragma unroll
          for (int e = 0; e < 8; ++e) w[cb][e] = f[e];
        }
      }
#pragma unroll
      for (int i = 0; i < LIN_MT; ++i) {
        const float4 xa = *reinterpret_cast<const float4*>(xs + i * Kp + k);
        const float4 xb = *reinterpret_cast<const float4*>(xs + i * Kp + k + 4);
        const float xv[8] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
#pragma unroll
        for (int cb = 0; cb < LIN_CB; ++cb)
#pragma unroll
          for (int e = 0; e < 8; ++e) acc[cb][i] = fmaf(xv[e], w[cb][e], acc[cb][i]);
      }
#pragma unroll
      for (int cb = 0; cb < LIN_CB; ++cb)
#pragma unroll
        for (int q = 0; q < RW; ++q) raw[cb][q] = nxt[cb][q];
    }
    for (int k = K8 + lane; k < K; k += 32) {
#pragma unroll
      for (int cb = 0; cb < LIN_CB; ++cb) {
        if (n0 + cb < N) {
          const long long off = static_cast<long long>(n0 + cb) * K + k;
          const float w = W_HALF ? __half2float(reinterpret_cast<const __half*>(Wv)[off])
                                 : reinterpret_cast<const float*>(Wv)[off];
#pragma unroll
          for (int i = 0; i < LIN_MT; ++i) acc[cb][i] = fmaf(xs[i * Kp + k], w, acc[cb][i]);
        }
      }
    }
#pragma unroll
    for (int cb = 0; cb < LIN_CB; ++cb) {
#pragma unroll
      for (int i = 0; i < LIN_MT; ++i) {
        float v = acc[cb][i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        const int n = n0 + cb;
        if (lane == 0 && i < mt && n < N) {
          if (b) v += b[n];
          if (silu_out) v = silu_f(v);
          if (add) v += add[static_cast<long long>(m0 + i) * ldadd + n];
          y[static_cast<long long>(m0 + i) * ldy + n] = v;
        }
      }
    }
  }
}

__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ x, const float* __restrict__ g,
                                                        const float* __restrict__ b, float* __restrict__ y, int N,
                                                        float eps) {
  __shared__ double sred[2][8];
  const int m = blockIdx.x;
  const float* xr = x + static_cast<long long>(m) * N;
  double s = 0.0, q = 0.0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    double v = xr[i];
    s += v;
    q += v * v;
  }
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    q += __shfl_xor_sync(0xffffffffu, q, o);
  }
  if ((threadIdx.x & 31) == 0) {
    sred[0][threadIdx.x >> 5] = s;
    sred[1][threadIdx.x >> 5] = q;
  }
  __syncthreads();
  s = 0.0;
  q = 0.0;
  for (int w = 0; w < 8; ++w) {
    s += sred[0][w];
    q += sred[1][w];
  }
  const double mean = s / N;
  double var = q / N - mean * mean;
  if (var < 0.0) var = 0.0;
  const float rstd = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
  const float fmean = static_cast<float>(mean);
  for (int i = threadIdx.x; i < N; i += blockDim.x)
    y[static_cast<long long>(m) * N + i] = (xr[i] - fmean) * rstd * g[i] + b[i];
}

// nn.py:101-121: [cos(t*f) | sin(t*f)], f_j = exp(-ln(max_period) * j / half), fp32
__global__ void timestep_embedding_kernel(const float* __restrict__ t, float* __restrict__ out, int B, int dim,
                                          float max_period) {
  const int half = dim / 2;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  pdl_wait();
  pdl_launch();
  if (i >= B * dim) return;
  const int b = i / dim, j = i % dim;
  float v = 0.f;
  if (j < 2 * half) {
    const int jj = j < half ? j : j - half;
    const float freq = expf(-logf(max_period) * static_cast<float>(jj) / static_cast<float>(half));
    const float arg = t[b] * freq;
    v = j < half ? cosf(arg) : sinf(arg);
  }
  out[i] = v;
}

__global__ void f32_to_f16_kernel(const float* __restrict__ x, __half* __restrict__ y, long long n) {
  long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (; i < n; i += stride) y[i] = __float2half_rn(x[i]);
}

// fp32 NCHW sources -> fp16 patch rows [NB*H*W, Kpad], k = tap*Cin + c
__global__ void __launch_bounds__(256) stem_im2col_kernel(const float* __restrict__ x, int Cx,
                                                          const float* __restrict__ x2, int C2,
                                                          const float* __restrict__ x3, int C3, int mul23, int NB,
                                                          int H, int W, __half* __restrict__ out, int Kpad) {
  const long long item = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(NB) * H * W * Kpad;
  pdl_wait();
  pdl_launch();
  if (item >= total) return;
  const int k = static_cast<int>(item % Kpad);
  const long long pix = item / Kpad;
  const int xx = static_cast<int>(pix % W);
  const int yy = static_cast<int>((pix / W) % H);
  const int n = static_cast<int>(pix / (static_cast<long long>(W) * H));
  const int Cin = Cx + C2 + C3;
  float v = 0.f;
  if (k < 9 * Cin) {
    const int tap = k / Cin, c = k % Cin;
    const int yi = yy + tap / 3 - 1, xi = xx + tap % 3 - 1;
    if (yi >= 0 && yi < H && xi >= 0 && xi < W) {
      const long long sp = static_cast<long long>(yi) * W + xi;
      if (c < Cx) {
        v = x[(static_cast<long long>(n) * Cx + c) * H * W + sp];
      } else if (c < Cx + C2) {
        v = x2[(static_cast<long long>(n) * C2 + (c - Cx)) * H * W + sp];
        if (mul23) v *= x3[static_cast<long long>(n) * C3 * H * W + sp];  // inpaint_image * inpaint_mask
      } else {
        v = x3[(static_cast<long long>(n) * C3 + (c - Cx - C2)) * H * W + sp];
      }
    }
  }
  out[item] = __float2half_rn(v);
}

// ------------------------------------------------------------------------------------------------
// sampler step
// ------------------------------------------------------------------------------------------------
struct SamplerParams {
  const float* model_out;  // [2B, 8, H, W]
  float* x;                // [B, 4, H, W]
  const float* noise;
  const float* coef;       // device [8]
  int B, HW;
  float guidance;
  int cond_first;
  float clip;
  int threshold_mode;
  const float* init;       // [B,4,H,W] or null
  const float* mask;       // [B,1,H,W] or null
  const float* rnoise;     // [B,4,H,W] or null: inpainting blends x_{t-1} with the re-noised init (diffusers) instead of x0
  float* x0;               // work [B*4*HW]
  float* sval;             // work scalar (dynamic threshold s)
};

__global__ void __launch_bounds__(256) sampler_x0_kernel(const SamplerParams p) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  pdl_wait();
  pdl_launch();
  const long long total = static_cast<long long>(p.B) * 4 * p.HW;
  if (i >= total) return;
  const int sp = static_cast<int>(i % p.HW);
  const int c = static_cast<int>((i / p.HW) % 4);
  const int b = static_cast<int>(i / (4LL * p.HW));
  const int bc = p.cond_first ? b : b + p.B;
  const int bu = p.cond_first ? b + p.B : b;
  const float ec = p.model_out[(static_cast<long long>(bc) * 8 + c) * p.HW + sp];
  const float eu = p.model_out[(static_cast<long long>(bu) * 8 + c) * p.HW + sp];
  const float eps = eu + p.guidance * (ec - eu);
  float x0 = p.coef[0] * p.x[i] - p.coef[1] * eps;
  x0 = fminf(fmaxf(x0, -p.clip), p.clip);
  if (p.mask && !p.rnoise) {  // Kandinsky 2.1: the known region replaces x0 (denoised_fun, kandinsky2_1_model.py:237-243)
    const float m = p.mask[static_cast<long long>(b) * p.HW + sp];
    x0 = x0 * (1.f - m) + p.init[i] * m;
  }
  p.x0[i] = x0;
}

// exact order statistics of |v[0..n)| (non-negative floats compare like their bit patterns):
// 4-pass byte radix select, single block. Reproduces np.percentile(|x|, 99.5) with linear interpolation, numpy >= 2
// semantics (gaussian_diffusion.py:288-292), and s = max(s, 1).
__device__ float radix_select(const float* __restrict__ v, int n, int rank, unsigned int* hist, unsigned int* sh) {
  unsigned int prefix = 0, mask = 0;
  int k = rank;
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const unsigned int u = __float_as_uint(fabsf(v[i]));
      if ((u & mask) == prefix) atomicAdd(&hist[(u >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned int cum = 0;
      int bin = 0;
      for (; bin < 256; ++bin) {
        if (cum + hist[bin] > static_cast<unsigned int>(k)) break;
        cum += hist[bin];
      }
      sh[0] = static_cast<unsigned int>(bin);
      sh[1] = cum;
    }
    __syncthreads();
    prefix |= sh[0] << shift;
    mask |= 255u << shift;
    k -= static_cast<int>(sh[1]);
    __syncthreads();
  }
  return __uint_as_float(prefix);
}

__global__ void __launch_bounds__(1024) sampler_percentile_kernel(const float* __restrict__ x0, int n, float* sval) {
  __shared__ unsigned int hist[256];
  __shared__ unsigned int sh[2];
  pdl_wait();
  pdl_launch();
  // numpy >= 2 on float32 data stays in float32 (NEP 50; numpy/lib/_function_base_impl.py): percentile divides q by
  // float32(100), the 'linear' virtual index is (n - 1) * q, _get_indexes takes floor / floor + 1 (both n - 1 when the index
  // reaches n - 1), _get_gamma is the exact fraction, and _lerp rounds every operation to float32.  The _rn intrinsics keep
  // nvcc from contracting any of these into an FMA.
  const float q = __fdiv_rn(99.5f, 100.0f);
  const float pos = __fmul_rn(static_cast<float>(n - 1), q);
  const bool top = pos >= static_cast<float>(n - 1);
  const int lo = top ? n - 1 : static_cast<int>(floorf(pos));
  const int hi = top ? n - 1 : lo + 1;
  const float a = radix_select(x0, n, lo, hist, sh);
  const float b = radix_select(x0, n, hi, hist, sh);
  if (threadIdx.x == 0) {
    // numpy _lerp: a + (b-a)*t, switched to b - (b-a)*(1-t) for t >= 0.5
    const float t = __fsub_rn(pos, static_cast<float>(lo));
    const float d = __fsub_rn(b, a);
    const float s = (t >= 0.5f) ? __fsub_rn(b, __fmul_rn(d, __fsub_rn(1.0f, t))) : __fadd_rn(a, __fmul_rn(d, t));
    *sval = fmaxf(s, 1.0f);
  }
}

__global__ void __launch_bounds__(256) sampler_post_kernel(const SamplerParams p) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  pdl_wait();
  pdl_launch();
  const long long total = static_cast<long long>(p.B) * 4 * p.HW;
  if (i >= total) return;
  const int sp = static_cast<int>(i % p.HW);
  const int c = static_cast<int>((i / p.HW) % 4);
  const int b = static_cast<int>(i / (4LL * p.HW));
  const int bc = p.cond_first ? b : b + p.B;
  float x0 = p.x0[i];
  if (p.threshold_mode == 1) {
    const float s = *p.sval;
    x0 = fminf(fmaxf(x0, -s), s) / s;
  }
  const float mean = p.coef[2] * x0 + p.coef[3] * p.x[i];
  const float v = p.model_out[(static_cast<long long>(bc) * 8 + 4 + c) * p.HW + sp];
  const float frac = (v + 1.f) * 0.5f;
  const float logvar = frac * p.coef[5] + (1.f - frac) * p.coef[4];
  float xp = mean + p.coef[6] * expf(0.5f * logvar) * p.noise[i];
  if (p.mask && p.rnoise) {
    // Kandinsky 2.2 (diffusers KandinskyV22InpaintPipeline): after the scheduler step the known region is replaced by the
    // clean latent noised to the NEXT timestep with the run's initial noise; coef[7] = sqrt(alphas_cumprod[t_next]), 1 at
    // the last step (which is also the pipeline's final blend with the clean latent)
    const float m = p.mask[static_cast<long long>(b) * p.HW + sp];
    const float c = p.coef[7];
    const float sgm = sqrtf(fmaxf(0.f, 1.f - c * c));
    xp = m * (c * p.init[i] + sgm * p.rnoise[i]) + (1.f - m) * xp;
  }
  p.x[i] = xp;
}

// PLMS / DDIM update with an explicit epsilon history (samplers.py:571-637):
//   e_t  = CFG(model_out)                                  (kandinsky2_1_model.py:222-233, eps channels only)
//   e'   = w[0]*e_t + w[1]*hist[0] + w[2]*hist[1] + w[3]*hist[2]      (Adams-Bashforth weights chosen by the host)
//   out  = sqrt(a_prev) * (x - sqrt(1-a_t) e') / sqrt(a_t) + sqrt(1-a_prev) e'      with coef = {1/sqrt(a_t),
//          sqrt(1-a_t)/sqrt(a_t), sqrt(a_prev), sqrt(1-a_prev)}
//   optionally e_t is stored into `store` (the history slot the host rotates in).
struct PlmsParams {
  const float* model_out;  // [2B, C2, H, W], eps = channels [0, 4)
  const float* x;          // [B, 4, H, W]
  float* out;              // [B, 4, H, W] (may alias x)
  const float* hist[3];
  float* store;            // or null
  const float* coef;       // device [8]: c0..c3 as above, w0..w3 = coef[4..8)
  int B, HW, C2;
  float guidance;
  int cond_first;
};

__global__ void __launch_bounds__(256) plms_step_kernel(const PlmsParams p) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  pdl_wait();
  pdl_launch();
  const long long total = static_cast<long long>(p.B) * 4 * p.HW;
  if (i >= total) return;
  const int sp = static_cast<int>(i % p.HW);
  const int c = static_cast<int>((i / p.HW) % 4);
  const int b = static_cast<int>(i / (4LL * p.HW));
  const int bc = p.cond_first ? b : b + p.B;
  const int bu = p.cond_first ? b + p.B : b;
  const float ec = p.model_out[(static_cast<long long>(bc) * p.C2 + c) * p.HW + sp];
  const float eu = p.model_out[(static_cast<long long>(bu) * p.C2 + c) * p.HW + sp];
  const float e_t = eu + p.guidance * (ec - eu);
  float ep = p.coef[4] * e_t;
  if (p.hist[0]) ep = fmaf(p.coef[5], p.hist[0][i], ep);
  if (p.hist[1]) ep = fmaf(p.coef[6], p.hist[1][i], ep);
  if (p.hist[2]) ep = fmaf(p.coef[7], p.hist[2][i], ep);
  const float x0 = p.coef[0] * p.x[i] - p.coef[1] * ep;
  const float xn = p.coef[2] * x0 + p.coef[3] * ep;
  if (p.store) p.store[i] = e_t;
  p.out[i] = xn;
}

// ------------------------------------------------------------------------------------------------
// MoVQ helpers
// ------------------------------------------------------------------------------------------------
// quntize.py:89-98: d = sum(z^2) + sum(e^2) - 2 z.e ; argmin (first minimum). dim == 4.
__global__ void __launch_bounds__(256) vq_argmin_kernel(const float* __restrict__ z, const float* __restrict__ cb,
                                                        long long* __restrict__ idx, int n, int n_embed) {
  extern __shared__ float4 scb[];  // tile of the codebook
  constexpr int TILE = 2048;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  float4 zv = make_float4(0.f, 0.f, 0.f, 0.f);
  if (i < n) zv = reinterpret_cast<const float4*>(z)[i];
  const float zz = ((zv.x * zv.x + zv.y * zv.y) + zv.z * zv.z) + zv.w * zv.w;
  float best = INFINITY;
  int bi = 0;
  for (int t0 = 0; t0 < n_embed; t0 += TILE) {
    const int cnt = min(TILE, n_embed - t0);
    __syncthreads();
    for (int j = threadIdx.x; j < cnt; j += blockDim.x) scb[j] = reinterpret_cast<const float4*>(cb)[t0 + j];
    __syncthreads();
    for (int j = 0; j < cnt; ++j) {
      const float4 e = scb[j];
      const float ee = ((e.x * e.x + e.y * e.y) + e.z * e.z) + e.w * e.w;
      const float dot = ((zv.x * e.x + zv.y * e.y) + zv.z * e.z) + zv.w * e.w;
      const float d = (zz + ee) - 2.f * dot;
      if (d < best) {
        best = d;
        bi = t0 + j;
      }
    }
  }
  if (i < n) idx[i] = bi;
}

__global__ void nchw_to_nhwc_f32_kernel(const float* __restrict__ x, float* __restrict__ y, int NB, int C, int H, int W) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(NB) * C * H * W;
  if (i >= total) return;
  const int c = static_cast<int>(i % C);
  const long long pix = i / C;
  const int sp = static_cast<int>(pix % (static_cast<long long>(H) * W));
  const int n = static_cast<int>(pix / (static_cast<long long>(H) * W));
  y[i] = x[(static_cast<long long>(n) * C + c) * H * W + sp];
}

// utils.py:57-70: ((x+1)*127.5).round().clamp(0,255).uint8, NCHW -> NHWC, cropped to (crop_h, crop_w)
__global__ void images_to_u8_kernel(const float* __restrict__ x, uint8_t* __restrict__ out, int NB, int C, int H, int W,
                                    int ch, int cw) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(NB) * ch * cw * C;
  if (i >= total) return;
  const int c = static_cast<int>(i % C);
  const long long pix = i / C;
  const int xx = static_cast<int>(pix % cw);
  const int yy = static_cast<int>((pix / cw) % ch);
  const int n = static_cast<int>(pix / (static_cast<long long>(cw) * ch));
  float v = (x[((static_cast<long long>(n) * C + c) * H + yy) * W + xx] + 1.f) * 127.5f;
  v = rintf(v);  // torch.round = round-half-to-even
  v = fminf(fmaxf(v, 0.f), 255.f);
  out[i] = static_cast<uint8_t>(v);
}

// tiny per-pixel channel mix on fp32 NCHW (MoVQ post_quant_conv 4->4, autoencoder.py:183)
__global__ void pointwise_nchw_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b,
                                      float* __restrict__ y, int NB, int Ci, int Co, int HW) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(NB) * Co * HW;
  if (i >= total) return;
  const int sp = static_cast<int>(i % HW);
  const int o = static_cast<int>((i / HW) % Co);
  const int n = static_cast<int>(i / (static_cast<long long>(HW) * Co));
  float acc = b ? b[o] : 0.f;
  for (int c = 0; c < Ci; ++c) acc = fmaf(w[o * Ci + c], x[(static_cast<long long>(n) * Ci + c) * HW + sp], acc);
  y[i] = acc;
}

// nearest 2x upsample of NHWC fp16 rows: one 16-byte vector per thread, each written to its 4 output pixels
__global__ void __launch_bounds__(256) upsample2x_kernel(const __half* __restrict__ x, int ldx, __half* __restrict__ y, int ldy,
                                                         int NB, int H, int W, int CV) {
  const long long item = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(NB) * H * W * CV;
  if (item >= total) return;
  const int v = static_cast<int>(item % CV);
  const long long pix = item / CV;
  const int xx = static_cast<int>(pix % W);
  const int yy = static_cast<int>((pix / W) % H);
  const int n = static_cast<int>(pix / (static_cast<long long>(W) * H));
  const uint4 val = __ldg(reinterpret_cast<const uint4*>(x + pix * ldx + v * 8));
#pragma unroll
  for (int dy = 0; dy < 2; ++dy)
#pragma unroll
    for (int dx = 0; dx < 2; ++dx) {
      const long long orow = (static_cast<long long>(n) * 2 * H + (2 * yy + dy)) * (2 * W) + (2 * xx + dx);
      *reinterpret_cast<uint4*>(y + orow * ldy + v * 8) = val;
    }
}

// every second pixel of NHWC fp16 rows: y[n, yo, xo, :] = x[n, 2*yo + oy, 2*xo + ox, :]
__global__ void __launch_bounds__(256) subsample2_kernel(const __half* __restrict__ x, int ldx, __half* __restrict__ y, int ldy,
                                                         int NB, int H, int W, int CV, int oy, int ox) {
  const int Ho = H / 2, Wo = W / 2;
  const long long item = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(NB) * Ho * Wo * CV;
  if (item >= total) return;
  const int v = static_cast<int>(item % CV);
  const long long pix = item / CV;
  const int xo = static_cast<int>(pix % Wo);
  const int yo = static_cast<int>((pix / Wo) % Ho);
  const int n = static_cast<int>(pix / (static_cast<long long>(Wo) * Ho));
  const long long irow = (static_cast<long long>(n) * H + (2 * yo + oy)) * W + (2 * xo + ox);
  *reinterpret_cast<uint4*>(y + pix * ldy + v * 8) = __ldg(reinterpret_cast<const uint4*>(x + irow * ldx + v * 8));
}

// row softmax, fp16 in/out, fp32 math; one block per row, 16-byte vectors
__global__ void __launch_bounds__(256) softmax_rows_kernel(const __half* __restrict__ x, int ldx, __half* __restrict__ y,
                                                           int ldy, int n, float scale_log2e) {
  __shared__ float red[8];
  const long long r = blockIdx.x;
  const __half* xr = x + r * ldx;
  __half* yr = y + r * ldy;
  const int nv = n / 8;
  float mx = -INFINITY;
  for (int v = threadIdx.x; v < nv; v += blockDim.x) {
    const uint4 raw = __ldg(reinterpret_cast<const uint4*>(xr + v * 8));
    const __half2* h2 = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = __half22float2(h2[e]);
      mx = fmaxf(mx, fmaxf(f.x, f.y));
    }
  }
  for (int i = nv * 8 + threadIdx.x; i < n; i += blockDim.x) mx = fmaxf(mx, __half2float(xr[i]));
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  mx = red[0];
  for (int w = 1; w < 8; ++w) mx = fmaxf(mx, red[w]);
  __syncthreads();
  const float mo = mx * scale_log2e;
  float sum = 0.f;
  for (int v = threadIdx.x; v < nv; v += blockDim.x) {
    const uint4 raw = __ldg(reinterpret_cast<const uint4*>(xr + v * 8));
    const __half2* h2 = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = __half22float2(h2[e]);
      sum += exp2f(fmaf(f.x, scale_log2e, -mo)) + exp2f(fmaf(f.y, scale_log2e, -mo));
    }
  }
  for (int i = nv * 8 + threadIdx.x; i < n; i += blockDim.x) sum += exp2f(fmaf(__half2float(xr[i]), scale_log2e, -mo));
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sum;
  __syncthreads();
  sum = 0.f;
  for (int w = 0; w < 8; ++w) sum += red[w];
  const float inv = 1.f / sum;
  for (int v = threadIdx.x; v < nv; v += blockDim.x) {
    const uint4 raw = __ldg(reinterpret_cast<const uint4*>(xr + v * 8));
    const __half2* h2 = reinterpret_cast<const __half2*>(&raw);
    uint4 ov;
    __half2* oh = reinterpret_cast<__half2*>(&ov);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = __half22float2(h2[e]);
      oh[e] = __floats2half2_rn(exp2f(fmaf(f.x, scale_log2e, -mo)) * inv, exp2f(fmaf(f.y, scale_log2e, -mo)) * inv);
    }
    *reinterpret_cast<uint4*>(yr + v * 8) = ov;
  }
  for (int i = nv * 8 + threadIdx.x; i < n; i += blockDim.x)
    yr[i] = __float2half_rn(exp2f(fmaf(__half2float(xr[i]), scale_log2e, -mo)) * inv);
}

inline unsigned int blocks_for(long long total, int bs) { return static_cast<unsigned int>((total + bs - 1) / bs); }

}  // namespace
}  // namespace k2

using namespace k2;

extern "C" {

int k2_linear(const float* x, int ldx, const void* W, int w_is_half, const float* b, const float* add, int ldadd,
              float* y, int ldy, int M, int N, int K, int silu_in, int silu_out, k2_stream_t stream) {
  K2_REQUIRE(x && W && y && M > 0 && N > 0 && K > 0, "linear: bad arguments");
  const int Kp = (K + 7) & ~7;
  const size_t smem = static_cast<size_t>(LIN_MT) * Kp * sizeof(float);
  K2_REQUIRE(smem <= 160 * 1024, "linear: K too large for the shared-memory x tile");
  const int vec_ok = ((K & 7) == 0) && ((reinterpret_cast<uintptr_t>(W) & 15) == 0);
  static bool attr_set = false;
  if (!attr_set) {
    K2_CHECK_CUDA(cudaFuncSetAttribute(linear_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    K2_CHECK_CUDA(cudaFuncSetAttribute(linear_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    attr_set = true;
  }
  const int ni = (N >= 8 * LIN_CB * LIN_NI * 2 * num_sms()) ? LIN_NI : 1;  // small N: keep every SM busy instead
  dim3 grid((N + 8 * LIN_CB * ni - 1) / (8 * LIN_CB * ni), (M + LIN_MT - 1) / LIN_MT);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (w_is_half)
    K2_CHECK_CUDA(launch_k(linear_kernel<true>, grid, dim3(256), smem, st, x, ldx, W, b, add, ldadd, y, ldy, M, N, K, Kp, vec_ok,
                           silu_in, silu_out, ni));
  else
    K2_CHECK_CUDA(launch_k(linear_kernel<false>, grid, dim3(256), smem, st, x, ldx, W, b, add, ldadd, y, ldy, M, N, K, Kp, vec_ok,
                           silu_in, silu_out, ni));
  K2_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int k2_layernorm(const float* x, const float* gamma, const float* beta, float* y, int M, int N, float eps,
                 k2_stream_t stream) {
  K2_REQUIRE(x && gamma && beta && y && M > 0 && N > 0, "layernorm: bad arguments");
  layernorm_kernel<<<M, 256, 0, static_cast<cudaStream_t>(stream)>>>(x, gamma, beta, y, N, eps);
  K2_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int k2_timestep_embedding(const float* t, float* out, int B, int dim, float max_period, k2_stream_t stream) {
  K2_REQUIRE(t && out && B > 0 && dim > 0, "timestep_embedding: bad arguments");
  K2_CHECK_CUDA(launch_k(timestep_embedding_kernel, dim3(blocks_for(static_cast<long long>(B) * dim, 256)), dim3(256), 0,
                         static_cast<cudaStream_t>(stream), t, out, B, dim, max_period));
  K2_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// SiLU on fp16, in place or out of place: the activations between the convolutions of the ControlNet hint stem (diffusers
// ImageHintTimeEmbedding.input_hint_block; once per generation, not on the per-step path)
static __global__ void __launch_bounds__(256) silu_f16_kernel(const __half2* __restrict__ x, __half2* __restrict__ y, long long n2) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n2;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float2 v = __half22float2(x[i]);
    y[i] = __floats2half2_rn(silu_f(v.x), silu_f(v.y));
  }
}

int k2_silu_f16(const void* x, void* y, long long n, k2_stream_t stream) {
  K2_REQUIRE(x && y && n > 0 && n % 2 == 0, "silu_f16: n must be a positive even element count");
  K2_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 3) == 0, "silu_f16: 4-byte alignment");
  long long blocks = (n / 2 + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  silu_f16_kernel<<<static_cast<unsigned int>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const __half2*>(x), reinterpret_cast<__half2*>(y), n / 2);
  K2_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int k2_f32_to_f16(const float* x, void* y, long long n, k2_stream_t stream) {
  K2_REQUIRE(x && y && n > 0, "f32_to_f16: bad arguments");
  long long blocks = (n + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  f32_to_f16_kernel<<<static_cast<unsigned int>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      x, reinterpret_cast<__half*>(y), n);
  K2_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int k2_stem_im2col(const float* x, int Cx, const float* x2, int C2, const float* x3, int C3, int mul23, int NB, int H,
                   int W, void* out, int Kpad, k2_stream_t stream) {
  K2_REQUIRE(x && out && Cx > 0, "stem_im2col: bad arguments");
  K2_REQUIRE(Kpad % 64 == 0 && Kpad >= 9 * (Cx + C2 + C3), "stem_im2col: Kpad too small / not a multiple of 64");
  K2_REQUIRE(!mul23 || (x2 && x3 && C3 == 1), "stem_im2col: mul23 needs x2 and a 1-channel x3");
  const long long total = static_cast<long long>(NB) * H * W * Kpad;
  K2_CHECK_CUDA(launch_k(stem_im2col_kernel, dim3(blocks_for(total, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream), x, Cx,
                         x2, C2, x3, C3, mul23, NB, H, W, reinterpret_cast<__half*>(out), Kpad));
  K2_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int k2_sampler_step(const float* model_out, float* x, const float* noise, const float* coef, int B, int H, int W,
                    float guidance, int cond_first, float clip, int threshold_mode, const float* inpaint_init,
                    const float* inpaint_mask, const float* inpaint_noise, float* work, k2_stream_t stream) {
  K2_REQUIRE(model_out && x && noise && coef && work && B > 0, "sampler_step: bad arguments");
  K2_REQUIRE((inpaint_init == nullptr) == (inpaint_mask == nullptr), "sampler_step: init and mask go together");
  K2_REQUIRE(inpaint_noise == nullptr || inpaint_init, "sampler_step: inpaint_noise without init / mask");
  SamplerParams p;
  p.model_out = model_out; p.x = x; p.noise = noise; p.coef = coef;
  p.B = B; p.HW = H * W; p.guidance = guidance; p.cond_first = cond_first; p.clip = clip;
  // threshold_mode: 0 clamp only; 1 dynamic threshold of LOCAL sample 0; 2 / 4 = first half of a split step (x0, and for 2 the
  // percentile of local sample 0) without the update; 3 = second half (update with the threshold found in `work`): lets a
  // sharded run broadcast the threshold of GLOBAL sample 0 between the halves (kandinsky2/model/gaussian_diffusion.py)
  K2_REQUIRE(threshold_mode >= 0 && threshold_mode <= 4, "sampler_step: threshold_mode in 0..4");
  const bool do_front = threshold_mode != 3;
  const bool do_pct = threshold_mode == 1 || threshold_mode == 2;
  const bool do_post = threshold_mode == 0 || threshold_mode == 1 || threshold_mode == 3;
  p.threshold_mode = (threshold_mode == 1 || threshold_mode == 3) ? 1 : 0;
  p.init = inpaint_init; p.mask = inpaint_mask; p.rnoise = inpaint_noise;
  p.x0 = work; p.sval = work + static_cast<long long>(B) * 4 * H * W;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long total = static_cast<long long>(B) * 4 * H * W;
  if (do_front) {
    K2_CHECK_CUDA(launch_k(sampler_x0_kernel, dim3(blocks_for(total, 256)), dim3(256), 0, st, p));
    count_launch();
  }
  if (do_pct) {
    K2_CHECK_CUDA(launch_k(sampler_percentile_kernel, dim3(1), dim3(1024), 0, st, static_cast<const float*>(p.x0), 4 * H * W,
                           p.sval));
    count_launch();
  }
  if (do_post) {
    K2_CHECK_CUDA(launch_k(sampler_post_kernel, dim3(blocks_for(total, 256)), dim3(256), 0, st, p));
    count_launch();
  }
  K2_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// Device-side schedule of the sampling loop (the whole denoising step is ONE CUDA graph, replayed once per step):
// step_begin reads the step counter k, duplicates the latent for classifier-free guidance, and stages this step's timestep,
// coefficient row and noise; step_end advances k.  Nothing comes from the host inside the loop.
__global__ void __launch_bounds__(256) step_begin_kernel(const float* __restrict__ x, float* __restrict__ x_in, long long n,
                                                         float* __restrict__ t_in, int nt, float* __restrict__ coef_out,
                                                         const float* __restrict__ ts_seq, const float* __restrict__ coef_seq,
                                                         const float* __restrict__ noise_seq, float* __restrict__ noise,
                                                         const int* __restrict__ counter) {
  pdl_wait();
  pdl_launch();
  const int k = counter[0] % max(counter[1], 1);  // counter = (step, steps in the schedule)
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) {
    const float v = x[i];
    x_in[i] = v;
    x_in[n + i] = v;
    if (noise_seq) noise[i] = noise_seq[static_cast<long long>(k) * n + i];
  }
  if (blockIdx.x == 0) {
    for (int j = threadIdx.x; j < nt; j += blockDim.x) t_in[j] = ts_seq[k];
    if (threadIdx.x < 8) coef_out[threadIdx.x] = coef_seq[k * 8 + threadIdx.x];
  }
}
__global__ void step_end_kernel(int* counter) {
  pdl_wait();
  pdl_launch();
  *counter += 1;
}

int k2_step_begin(const float* x, float* x_in, long long n, float* t_in, int nt, float* coef_out, const float* ts_seq,
                  const float* coef_seq, const float* noise_seq, float* noise, const int* counter, k2_stream_t stream) {
  K2_REQUIRE(x && x_in && t_in && coef_out && ts_seq && coef_seq && counter && n > 0 && nt > 0, "step_begin: bad arguments");
  K2_REQUIRE((noise_seq == nullptr) || noise, "step_begin: noise_seq without a noise buffer");
  K2_CHECK_CUDA(launch_k(step_begin_kernel, dim3(blocks_for(n, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream), x, x_in, n,
                         t_in, nt, coef_out, ts_seq, coef_seq, noise_seq, noise, counter));
  count_launch();
  return 0;
}

int k2_step_end(int* counter, k2_stream_t stream) {
  K2_REQUIRE(counter, "step_end: null counter");
  K2_CHECK_CUDA(launch_k(step_end_kernel, dim3(1), dim3(1), 0, static_cast<cudaStream_t>(stream), counter));
  count_launch();
  return 0;
}

int k2_upsample2x_nhwc(const void* x, int ldx, void* y, int ldy, int NB, int H, int W, int C, k2_stream_t stream) {
  K2_REQUIRE(x && y && C % 8 == 0 && ldx % 8 == 0 && ldy % 8 == 0, "upsample2x: channels / strides must be multiples of 8");
  const long long total = static_cast<long long>(NB) * H * W * (C / 8);
  upsample2x_kernel<<<blocks_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const __half*>(x), ldx, reinterpret_cast<__half*>(y), ldy, NB, H, W, C / 8);
  K2_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int k2_subsample2_nhwc(const void* x, int ldx, void* y, int ldy, int NB, int H, int W, int C, int oy, int ox,
                       k2_stream_t stream) {
  K2_REQUIRE(x && y && C % 8 == 0 && ldx % 8 == 0 && ldy % 8 == 0 && H % 2 == 0 && W % 2 == 0 && (oy | 1) == 1 && (ox | 1) == 1,
             "subsample2: bad arguments");
  const long long total = static_cast<long long>(NB) * (H / 2) * (W / 2) * (C / 8);
  subsample2_kernel<<<blocks_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const __half*>(x), ldx, reinterpret_cast<__half*>(y), ldy, NB, H, W, C / 8, oy, ox);
  K2_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int k2_softmax_rows(const void* x, int ldx, void* y, int ldy, long long rows, int n, float scale, k2_stream_t stream) {
  K2_REQUIRE(x && y && rows > 0 && n > 0 && ldx % 8 == 0 && ldy % 8 == 0, "softmax_rows: bad arguments");
  K2_REQUIRE(rows < (1LL << 31), "softmax_rows: too many rows");
  softmax_rows_kernel<<<static_cast<unsigned int>(rows), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const __half*>(x), ldx, reinterpret_cast<__half*>(y), ldy, n, scale * 1.4426950408889634f);
  K2_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int k2_plms_step(const float* model_out, int C2, const float* x, float* out, const float* hist0, const float* hist1,
                 const float* hist2, float* store, const float* coef, int B, int H, int W, float guidance, int cond_first,
                 k2_stream_t stream) {
  K2_REQUIRE(model_out && x && out && coef && B > 0 && C2 >= 4, "plms_step: bad arguments");
  PlmsParams p;
  p.model_out = model_out; p.x = x; p.out = out; p.hist[0] = hist0; p.hist[1] = hist1; p.hist[2] = hist2; p.store = store;
  p.coef = coef; p.B = B; p.HW = H * W; p.C2 = C2; p.guidance = guidance; p.cond_first = cond_first;
  const long long total = static_cast<long long>(B) * 4 * H * W;
  K2_CHECK_CUDA(launch_k(plms_step_kernel, dim3(blocks_for(total, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream), p));
  count_launch();
  return 0;
}

int k2_vq_argmin(const float* z, const float* codebook, long long* idx, int n, int n_embed, int dim,
                 k2_stream_t stream) {
  K2_REQUIRE(z && codebook && idx && n > 0 && n_embed > 0, "vq_argmin: bad arguments");
  K2_REQUIRE(dim == 4, "vq_argmin: only embed_dim 4 (MoVQ) is implemented");
  vq_argmin_kernel<<<blocks_for(n, 256), 256, 2048 * sizeof(float4), static_cast<cudaStream_t>(stream)>>>(
      z, codebook, idx, n, n_embed);
  K2_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int k2_nchw_to_nhwc_f32(const float* x, float* y, int NB, int C, int H, int W, k2_stream_t stream) {
  K2_REQUIRE(x && y, "nchw_to_nhwc: null");
  nchw_to_nhwc_f32_kernel<<<blocks_for(static_cast<long long>(NB) * C * H * W, 256), 256, 0,
                            static_cast<cudaStream_t>(stream)>>>(x, y, NB, C, H, W);
  K2_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int k2_images_to_u8(const float* x_nchw, uint8_t* out_nhwc, int NB, int C, int H, int W, int crop_h, int crop_w,
                    k2_stream_t stream) {
  K2_REQUIRE(x_nchw && out_nhwc && crop_h <= H && crop_w <= W, "images_to_u8: bad arguments");
  images_to_u8_kernel<<<blocks_for(static_cast<long long>(NB) * crop_h * crop_w * C, 256), 256, 0,
                        static_cast<cudaStream_t>(stream)>>>(x_nchw, out_nhwc, NB, C, H, W, crop_h, crop_w);
  K2_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int k2_pointwise_nchw_f32(const float* x, const float* w, const float* b, float* y, int NB, int Ci, int Co, int HW,
                          k2_stream_t stream) {
  K2_REQUIRE(x && w && y && Ci > 0 && Co > 0, "pointwise_nchw: bad arguments");
  pointwise_nchw_kernel<<<blocks_for(static_cast<long long>(NB) * Co * HW, 256), 256, 0,
                          static_cast<cudaStream_t>(stream)>>>(x, w, b, y, NB, Ci, Co, HW);
  K2_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

}  // extern "C"
