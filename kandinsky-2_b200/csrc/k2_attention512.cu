// k2_attention512.cu -- fused softmax(q k^T / sqrt(C)) v for ONE head of width C = 512 on tcgen05 tensor cores: the MoVQ
// AttnBlock (kandinsky2/vqgan/movq_modules.py:201-225; encoder twin vqgan_blocks.py:186-240) without the [T, T] score matrix
// in HBM (680 MB for four 768 x 768 images, written once and read twice by the unfused path).
//
// The constraint that shapes the kernel is TMEM: an fp32 accumulator for O[128 queries, 512 channels] alone is all 512
// columns, and S needs 128 more.  So a CTA owns 128 queries and HALF of the output channels (256 columns of O + two
// 128-column S buffers = 512), and the two CTAs of a query tile both compute the full score tile: 1.5x the attention MACs
// (the QK^T product twice), in exchange for never materialising the scores.
//
//   per CTA: Q[128, 512] resident in shared memory (8 K-major swizzle atoms of 16 KB)
//   per 128-key block j:   S(j)   = Q K(j)^T      8 d-chunks x (M128 N128 K64)   -> TMEM S[j & 1]
//                          P(j)   = exp2(S*c - m) one softmax thread per query row (128 scores), two passes over TMEM:
//                                   row maximum first, then the exponentials -> fp16 pairs -> TENSOR memory, written over
//                                   the first 64 columns of the very S buffer they came from (chunk c of P lands on
//                                   columns the thread has already consumed)
//                          O     += P(j) V(j)     4 d-chunks (of this CTA's half) x (M128 N64 K128), A operand = P from
//                                                 tensor memory (tcgen05.mma [d], [a], b-desc), V used MN-major as TMA
//                                                 lands it, O rescaled lazily (only when a row maximum grows by 2^8)
//   Shared-memory operand reads per key block: S 256 KB + V 64 KB.  With P in shared memory (round-2 first version) the PV
//   product re-read the 32 KB P tile for each of the four V chunks: 448 KB per block at 128 B/clk = 3500 cycles, exactly the
//   measured 3584 -- the kernel was shared-memory-bandwidth bound, not tensor bound (3072 cycles of MMA per block).
//   S(j+2) reuses the buffer of S(j) / P(j): it is issued after PV(j), and the tensor pipe executes in issue order, so no
//   barrier is needed for that hand-back.
//   K / V chunks (128 keys x 64 channels = 16 KB) stream through ONE 6-stage ring in the order the MMA warp consumes them:
//   K(0); then K(j+1), V(j) per block, so S(j+1) is being produced while the softmax of block j runs.
// Warp roles (256 threads): warp 0 TMA producer, warp 1 MMA issuer, warp 2 TMEM allocator, warps 4-7 softmax + epilogue.
#include <string.h>

#include <algorithm>

#include "../../include/k2b200.h"
#include "k2_common.cuh"
#include "k2_internal.h"

namespace k2 {
namespace {

constexpr int BQ = 128;                  // queries per CTA
constexpr int BKV = 128;                 // keys per block
constexpr int DC = 64;                   // channels per chunk (one 128-byte swizzle row)
constexpr int CH = 512;                  // head width
constexpr int NQC = CH / DC;             // 8 chunks of Q / K along the channels
constexpr int OH = 256;                  // output channels per CTA
constexpr int NVC = OH / DC;             // 4 V chunks per block
constexpr int TILE_BYTES = 128 * DC * 2; // 16 KB
constexpr int STAGES = 6;
constexpr int SMEM_Q = 0;
constexpr int SMEM_RING = SMEM_Q + NQC * TILE_BYTES;        // 128 KB
constexpr int SMEM_BAR = SMEM_RING + STAGES * TILE_BYTES;   // + 96 KB
constexpr int SMEM_TOTAL = SMEM_BAR + 256 + 1024;           // barriers + alignment slack = 230,656 B <= 232,448
constexpr int TM_S = 0;                  // S buffer b at columns b * 128; P(j) over columns [0, 64) of S[j & 1]
constexpr int TM_O = 256;                // O: 256 columns
constexpr float RESCALE_GAP = 8.f;

struct Attn512Params {
  CUtensorMap tm;        // 3-D (channels, T, B) over the qkv rows, box (64, 128, 1)
  int B, T;
  int q_off, k_off, v_off;
  __half* out;           // [B, T, ldo]
  int ldo;
  float scale_log2e;
};

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__global__ void __launch_bounds__(256, 1) attention_d512_kernel(const __grid_constant__ Attn512Params p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SMEM_BAR);
  uint64_t* q_full = bars;                 // 1
  uint64_t* ring_full = bars + 1;          // STAGES
  uint64_t* ring_empty = ring_full + STAGES;
  uint64_t* s_full = ring_empty + STAGES;  // 2
  uint64_t* p_full = s_full + 2;           // 1
  uint64_t* pv_done = p_full + 1;          // 1
  // the epilogue cannot wait for PV(nblk - 1) by pv_done's parity: the common path never waits for PV(j), so when the softmax
  // of the last block ends, PV(nblk - 2) may still be pending, and its phase has the parity of the one the epilogue wants
  uint64_t* o_full = pv_done + 1;          // 1: committed once, after the last PV product
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(o_full + 1);

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * BQ;
  const int dh = blockIdx.y;               // which half of the output channels
  const int b = blockIdx.z;
  const int nblk = (p.T + BKV - 1) / BKV;

  if (warp_idx == 0 && lane == 0) tma_prefetch_desc(&p.tm);
  if (warp_idx == 1 && lane == 0) {
    mbar_init(q_full, 1);
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&ring_full[i], 1);
      mbar_init(&ring_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s_full[i], 1);
    }
    mbar_init(p_full, 4);
    mbar_init(pv_done, 1);
    mbar_init(o_full, 1);
    fence_barrier_init();
  }
  if (warp_idx == 2) {
    tmem_alloc(tmem_ptr, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  pdl_wait();
  pdl_launch();

  if (warp_idx == 0) {
    // ===================================== TMA producer =====================================
    if (elect_one()) {
      mbar_arrive_expect_tx(q_full, NQC * TILE_BYTES);
      for (int c = 0; c < NQC; ++c) tma_load_3d(smem + SMEM_Q + c * TILE_BYTES, &p.tm, q_full, p.q_off + c * DC, q0, b);
      int stage = 0;
      uint32_t phase = 0;
      auto push = [&](int chan, int row) {
        mbar_wait(&ring_empty[stage], phase ^ 1);
        mbar_arrive_expect_tx(&ring_full[stage], TILE_BYTES);
        tma_load_3d(smem + SMEM_RING + stage * TILE_BYTES, &p.tm, &ring_full[stage], chan, row, b);
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      };
      for (int c = 0; c < NQC; ++c) push(p.k_off + c * DC, 0);
      for (int j = 0; j < nblk; ++j) {
        if (j + 1 < nblk)
          for (int c = 0; c < NQC; ++c) push(p.k_off + c * DC, (j + 1) * BKV);
        for (int c = 0; c < NVC; ++c) push(p.v_off + dh * OH + c * DC, j * BKV);
      }
    }
  } else if (warp_idx == 1) {
    // ===================================== MMA issuer ========================================
    if (elect_one()) {
      constexpr uint32_t idesc_s = make_idesc_f16(BQ, BKV, 0, 0);  // Q (K-major) x K (K-major)
      constexpr uint32_t idesc_o = make_idesc_f16(BQ, DC, 0, 1);   // P (K-major, tensor memory) x V (MN-major), N = 64
      int stage = 0;
      uint32_t phase = 0;
      auto next_stage = [&]() {
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      };
      auto issue_s = [&](int jb) {  // S[jb & 1] = Q K(jb)^T over the 8 channel chunks
        const uint32_t d = tmem_base + TM_S + (jb & 1) * BKV;
        for (int c = 0; c < NQC; ++c) {
          mbar_wait(&ring_full[stage], phase);
          tc_fence_after();
          const uint64_t adesc = make_sw128_desc(smem_u32(smem + SMEM_Q + c * TILE_BYTES));
          const uint64_t bdesc = make_sw128_desc(smem_u32(smem + SMEM_RING + stage * TILE_BYTES));
#pragma unroll
          for (int k = 0; k < DC / 16; ++k)
            umma_f16(d, adesc + static_cast<uint64_t>(k * 2), bdesc + static_cast<uint64_t>(k * 2), idesc_s, (c | k) != 0 ? 1u : 0u);
          umma_commit(&ring_empty[stage]);
          next_stage();
        }
        umma_commit(&s_full[jb & 1]);
      };
      mbar_wait(q_full, 0);
      tc_fence_after();
      issue_s(0);
      for (int j = 0; j < nblk; ++j) {
        // S[(j+1) & 1] last held S(j-1) / P(j-1): the softmax warps finished with it before p_full(j-1), and PV(j-1) was
        // issued in the previous iteration -- the tensor pipe retires it before this product starts
        if (j + 1 < nblk) issue_s(j + 1);
        mbar_wait(p_full, j & 1);
        tc_fence_after();
        const uint32_t p_tm = tmem_base + TM_S + (j & 1) * BKV;
        for (int c = 0; c < NVC; ++c) {
          mbar_wait(&ring_full[stage], phase);
          tc_fence_after();
          const uint32_t v_addr = smem_u32(smem + SMEM_RING + stage * TILE_BYTES);
          const uint32_t d = tmem_base + TM_O + c * DC;
#pragma unroll
          for (int k = 0; k < BKV / 16; ++k) {
            // A: P from tensor memory, 16 keys = 8 columns of fp16 pairs per step
            // B: V chunk [128 keys][64 channels] (MN-major): 16 keys = 16 rows of 128 B = 2048 B per step
            const uint64_t bdesc = make_sw128_desc(v_addr + k * 2048);
            umma_f16_ts(d, p_tm + k * 8, bdesc, idesc_o, (j > 0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&ring_empty[stage]);
          next_stage();
        }
        umma_commit(pv_done);
      }
      umma_commit(o_full);
    }
  } else if (warp_idx >= 4) {
    // ===================================== softmax + epilogue =================================
    const int ew = warp_idx & 3;                  // TMEM lane quarter
    const int row = ew * 32 + lane;               // query row == TMEM lane
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16);
    const uint32_t o_addr = lane_addr + TM_O;
    const float c = p.scale_log2e;
    float m_used = 0.f, l_run = 0.f;
    for (int j = 0; j < nblk; ++j) {
      const uint32_t s_addr = lane_addr + TM_S + (j & 1) * BKV;
      const int valid = min(BKV, p.T - j * BKV);
      mbar_wait(&s_full[j & 1], (j >> 1) & 1);
      tc_fence_after();
      // pass 1: row maximum (scores stay in TMEM; reading them twice is cheaper than 128 live registers)
      float mx = -INFINITY;
#pragma unroll
      for (int part = 0; part < 4; ++part) {
        uint32_t s[32];
        tmem_ld_32x32b_x32(s_addr + part * 32, s);
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < 32; e += 2) {
          const float a0 = (part * 32 + e < valid) ? __uint_as_float(s[e]) : -INFINITY;
          const float a1 = (part * 32 + e + 1 < valid) ? __uint_as_float(s[e + 1]) : -INFINITY;
          mx = fmax3(mx, a0, a1);
        }
      }
      const float m_blk = mx * c;
      if (j == 0) {
        m_used = m_blk;
      } else {
        const bool grow = m_blk > m_used + RESCALE_GAP;
        if (__any_sync(0xffffffffu, grow)) {
          // rare path: O must hold every block < j before it is rescaled.  (The common path needs no wait at all: P(j)
          // goes into S(j)'s own buffer, and S(j) was produced after PV(j-2) released it.)
          mbar_wait(pv_done, (j - 1) & 1);
          tc_fence_after();
          const float m_new = grow ? m_blk : m_used;
          const float alpha = ex2f(m_used - m_new);
#pragma unroll 1
          for (int oc = 0; oc < OH; oc += 32) {
            uint32_t o[32];
            tmem_ld_32x32b_x32(o_addr + oc, o);
            tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 32; ++e) o[e] = __float_as_uint(__uint_as_float(o[e]) * alpha);
            tmem_st_32x32b_x32(o_addr + oc, o);
          }
          tmem_st_wait();
          l_run *= alpha;
          m_used = m_new;
        }
      }
      // pass 2: P = exp2(S*c - m_used) -> fp16 -> the K-major swizzled A operand of the PV product
      float l0 = 0.f, l1 = 0.f;
#pragma unroll
      for (int part = 0; part < 4; ++part) {
        uint32_t s[32];
        tmem_ld_32x32b_x32(s_addr + part * 32, s);
        tmem_ld_wait();
        uint32_t packed[16];
#pragma unroll
        for (int e = 0; e < 32; e += 2) {
          float p0 = ex2f(fmaf(__uint_as_float(s[e]), c, -m_used));
          float p1 = ex2f(fmaf(__uint_as_float(s[e + 1]), c, -m_used));
          if (part * 32 + e >= valid) p0 = 0.f;
          if (part * 32 + e + 1 >= valid) p1 = 0.f;
          l0 += p0;
          l1 += p1;
          __half2 hh = __floats2half2_rn(p0, p1);
          packed[e >> 1] = *reinterpret_cast<uint32_t*>(&hh);
        }
        // keys 2c, 2c+1 of the block -> column c of S[j & 1]: chunk `part` covers columns [16 part, 16 part + 16), all of
        // them inside score columns this thread has already pulled into registers
        tmem_st_32x32b_x16(s_addr + part * 16, packed);
      }
      l_run += l0 + l1;
      // P(j) complete in tensor memory -> let the MMA warp go
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full);
    }
    // epilogue: O / l -> fp16, each thread writes the 256 channels of its row (512 contiguous bytes)
    mbar_wait(o_full, 0);
    tc_fence_after();
    const int q = q0 + row;
    const float inv = 1.f / l_run;
    __half* orow = p.out + (static_cast<long long>(b) * p.T + q) * p.ldo + dh * OH;
#pragma unroll 1
    for (int oc = 0; oc < OH; oc += 32) {
      uint32_t o[32];
      tmem_ld_32x32b_x32(o_addr + oc, o);
      tmem_ld_wait();
      if (q < p.T) {
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          uint4 ov;
          __half2* oh = reinterpret_cast<__half2*>(&ov);
#pragma unroll
          for (int e = 0; e < 4; ++e)
            oh[e] = __floats2half2_rn(__uint_as_float(o[v * 8 + 2 * e]) * inv, __uint_as_float(o[v * 8 + 2 * e + 1]) * inv);
          *reinterpret_cast<uint4*>(orow + oc + v * 8) = ov;
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp_idx == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace
}  // namespace k2

using namespace k2;

extern "C" int k2_attention_d512(const void* qkv, int ldq, int q_off, int k_off, int v_off, int B, int T, float scale, void* out,
                                 int ldo, k2_stream_t stream) {
  K2_REQUIRE(qkv && out && B > 0 && T > 0, "attention_d512: bad arguments");
  K2_REQUIRE(ldq % 8 == 0 && ldo % 8 == 0 && q_off % 8 == 0 && k_off % 8 == 0 && v_off % 8 == 0 && ldo >= CH,
             "attention_d512: strides / offsets must be multiples of 8 elements");
  K2_REQUIRE(std::max(std::max(q_off, k_off), v_off) + CH <= ldq, "attention_d512: qkv row narrower than the offsets + 512");
  K2_REQUIRE((reinterpret_cast<uintptr_t>(qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
             "attention_d512: 16-byte alignment");
  Attn512Params p;
  memset(&p, 0, sizeof p);
  {
    uint64_t dims[3] = {static_cast<uint64_t>(ldq), static_cast<uint64_t>(T), static_cast<uint64_t>(B)};
    uint64_t str[2] = {static_cast<uint64_t>(ldq) * 2, static_cast<uint64_t>(ldq) * 2 * T};
    uint32_t box[3] = {64, 128, 1};
    if (encode_tmap_f16(&p.tm, qkv, 3, dims, str, box)) return -1;
  }
  p.B = B; p.T = T; p.q_off = q_off; p.k_off = k_off; p.v_off = v_off;
  p.out = reinterpret_cast<__half*>(out);
  p.ldo = ldo;
  p.scale_log2e = scale * 1.4426950408889634f;
  static bool attr_set = false;
  if (!attr_set) {
    K2_CHECK_CUDA(cudaFuncSetAttribute(attention_d512_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_TOTAL));
    attr_set = true;
  }
  dim3 grid((T + BQ - 1) / BQ, 2, B);
  K2_CHECK_CUDA(launch_k(attention_d512_kernel, grid, dim3(256), SMEM_TOTAL, static_cast<cudaStream_t>(stream), p));
  count_launch();
  return 0;
}
