// Flash-style fused attention on tcgen05: S = Q K^T and O += P V on the tensor cores with S, O in TMEM,
// online softmax in registers (one query row per thread), lazy rescale of O (only when the running max
// moves by more than 2^8), P staged through swizzled shared memory as the A operand of the second MMA.
//
//   warp 0     : TMA producer (Q once; K / V^T tiles double-buffered)
//   warp 1     : TMEM alloc + tcgen05.mma issue: S(j+1) is issued before PV(j) so softmax(j+1) overlaps PV(j)
//   warps 2..5 : softmax / correction / epilogue (128 query rows)
//
// Replaces the materialised einsum('b i d, b j d -> b i j') * scale -> softmax -> einsum('b i j, b j d -> b i d')
// of ldm/modules/attention.py:178-192 (and CLIP self-attention with a causal mask).
#include "../../include/sdb200.h"
#include "host.h"
#include "ptx.cuh"

#include <stdlib.h>

namespace sdb {

constexpr int AQ = 128;   // query rows per CTA
constexpr int AKV = 64;   // kv rows per iteration
// K / V^T ring depth. The next K tile can only be requested once the PV MMA that last read the slot has finished, so
// with 2 slots the ~1 us TMA round trip sat on the per-iteration critical path (155 us for N=4096, d=40); 3 slots take
// it off (DPAD 192 keeps 2: shared memory).
template <int DPAD>
struct AttnCfg {
  static constexpr int ST = DPAD <= 128 ? 3 : 2;
  static constexpr int SMEM = AQ * DPAD * 2 + ST * (2 * AKV * DPAD * 2) + 2 * AQ * AKV * 2 + 1024;
};

struct AttnArgs {
  int nq, nkv, d, heads;
  int ldo;
  long long o_batch_stride;
  __half* out;
  float scale_log2;
  int causal;
};

__device__ __forceinline__ float fast_exp2(float x) {  // one MUFU.EX2, flush-to-zero (exp2(-inf) = 0)
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <int DPAD>
__global__ void __launch_bounds__(192)
    attention_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                        const __grid_constant__ CUtensorMap tmV, const AttnArgs p) {
  constexpr int PANELS = DPAD / 64;
  constexpr int Q_BYTES = AQ * DPAD * 2;
  constexpr int K_BYTES = AKV * DPAD * 2;
  constexpr int V_BYTES = DPAD * AKV * 2;
  constexpr int P_BYTES = AQ * AKV * 2;
  constexpr int TMEM_COLS = (128 + DPAD) <= 256 ? 256 : 512;
  constexpr int ST = AttnCfg<DPAD>::ST;
  constexpr uint32_t O_COL = 128;

  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment by offset (keeps the shared address space visible to the compiler: STS, not generic ST)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* q_s = smem;
  uint8_t* k_s = q_s + Q_BYTES;        // ST stages
  uint8_t* v_s = k_s + ST * K_BYTES;   // ST stages
  uint8_t* p_s = v_s + ST * V_BYTES;   // 2 buffers

  __shared__ uint64_t q_full, k_full[ST], v_full[ST], kv_empty[ST], s_full[2], p_full[2], pv_done[2];
  __shared__ uint32_t tmem_base_smem;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  pdl_launch_dependents();
  const int q0 = blockIdx.x * AQ;
  const int head = blockIdx.y;
  const int b = blockIdx.z;
  int nkv_eff = p.nkv;
  if (p.causal) nkv_eff = min(p.nkv, q0 + AQ);  // kv blocks entirely above the diagonal are skipped
  const int n_iter = (nkv_eff + AKV - 1) / AKV;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    mbar_init(&q_full, 1);
    for (int i = 0; i < ST; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&v_full[i], 1);
      mbar_init(&kv_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&p_full[i], 128);
      mbar_init(&pv_done[i], 1);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(&tmem_base_smem, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_smem;

  pdl_wait();   // q / k / v come from the previous kernels; everything above overlapped their tail
  if (warp == 0) {
    if (elect_one()) {
      mbar_arrive_expect_tx(&q_full, Q_BYTES);
      for (int pn = 0; pn < PANELS; ++pn)
        tma_load_3d(q_s + pn * (AQ * 128), &tmQ, &q_full, head * DPAD + pn * 64, q0, b);
      for (int j = 0; j < n_iter; ++j) {
        int s = j % ST;
        uint32_t ph = (j / ST) & 1;
        mbar_wait(&kv_empty[s], ph ^ 1);
        mbar_arrive_expect_tx(&k_full[s], K_BYTES);
        for (int pn = 0; pn < PANELS; ++pn)
          tma_load_3d(k_s + s * K_BYTES + pn * (AKV * 128), &tmK, &k_full[s], head * DPAD + pn * 64, j * AKV, b);
        mbar_arrive_expect_tx(&v_full[s], V_BYTES);
        tma_load_3d(v_s + s * V_BYTES, &tmV, &v_full[s], j * AKV, head * DPAD, b);
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc_s = umma_idesc_f16(AQ, AKV);
      // head dimension d < DPAD: columns d .. DPAD-1 of Q / K and rows d .. DPAD-1 of V^T are zero padding. Only the
      // 16-wide K steps that hold real columns are issued for S, and O is accumulated ceil16(d) columns wide: the
      // tensor pipe (and the TMEM port it blocks for the softmax warps' loads) is busy d/DPAD of the time it was
      const int ksteps = (p.d + 15) >> 4;
      const uint32_t idesc_o = umma_idesc_f16(AQ, ksteps * 16);
      const uint32_t q_addr = smem_u32(q_s);
      auto issue_s = [&](int j) {
        const int s = j & 1;            // S accumulator buffer
        const int ks = j % ST;          // K/V ring slot
        mbar_wait(&k_full[ks], (j / ST) & 1);
        tc_fence_after();
        const uint32_t k_addr = smem_u32(k_s + ks * K_BYTES);
#pragma unroll
        for (int kk = 0; kk < DPAD / 16; ++kk) {
          if (kk >= ksteps) break;
          uint64_t da = umma_desc_k128(q_addr + (kk >> 2) * (AQ * 128) + (kk & 3) * 32);
          uint64_t db = umma_desc_k128(k_addr + (kk >> 2) * (AKV * 128) + (kk & 3) * 32);
          umma_f16(tmem + s * AKV, da, db, idesc_s, kk > 0 ? 1u : 0u);
        }
        umma_commit(&s_full[s]);
      };
      mbar_wait(&q_full, 0);
      if (n_iter > 0) issue_s(0);
      for (int j = 0; j < n_iter; ++j) {
        int s = j & 1;
        uint32_t ph = (j >> 1) & 1;
        if (j + 1 < n_iter) issue_s(j + 1);
        const int ks = j % ST;
        mbar_wait(&p_full[s], ph);
        mbar_wait(&v_full[ks], (j / ST) & 1);
        tc_fence_after();
        const uint32_t p_addr = smem_u32(p_s + s * P_BYTES);
        const uint32_t v_addr = smem_u32(v_s + ks * V_BYTES);
#pragma unroll
        for (int kk = 0; kk < AKV / 16; ++kk) {
          uint64_t da = umma_desc_k128(p_addr + kk * 32);
          uint64_t db = umma_desc_k128(v_addr + kk * 32);
          umma_f16(tmem + O_COL, da, db, idesc_o, (j > 0 || kk > 0) ? 1u : 0u);
        }
        umma_commit(&kv_empty[ks]);
        umma_commit(&pv_done[s]);
      }
    }
  } else {
    const int lg = warp & 3;
    const int r = lg * 32 + lane;
    const int qi = q0 + r;
    const uint32_t lane_addr = static_cast<uint32_t>(lg * 32) << 16;
    float m_used = -INFINITY;
    float l = 0.f;
    for (int j = 0; j < n_iter; ++j) {
      const int s = j & 1;
      mbar_wait(&s_full[s], (j >> 1) & 1);
      tc_fence_after();
      float t[AKV];  // raw scores q.k (unscaled); the softmax scale is folded into one FFMA per element below
      {
        uint32_t r0[32], r1[32];
        tmem_ld32(tmem + lane_addr + s * AKV, r0);
        tmem_ld32(tmem + lane_addr + s * AKV + 32, r1);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < 32; ++c) {
          t[c] = __uint_as_float(r0[c]);
          t[32 + c] = __uint_as_float(r1[c]);
        }
      }
      const int kv0 = j * AKV;
      // only the ragged last block and (causal) diagonal blocks need per-element masking
      if ((kv0 + AKV > p.nkv) || (p.causal && kv0 + AKV - 1 > q0)) {
#pragma unroll
        for (int c = 0; c < AKV; ++c) {
          int kv = kv0 + c;
          if ((kv >= p.nkv) || (p.causal && kv > qi)) t[c] = -INFINITY;
        }
      }
      // 8 independent partial maxima / sums: a serial 64-deep FMNMX / FADD chain would expose ~4 cycles per element
      // with only two softmax warps per scheduler to hide it
      float mx[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) mx[i] = t[i];
#pragma unroll
      for (int c = 8; c < AKV; ++c) mx[c & 7] = fmaxf(mx[c & 7], t[c]);
      const float m_raw = fmaxf(fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3])), fmaxf(fmaxf(mx[4], mx[5]), fmaxf(mx[6], mx[7])));
      const float m_blk = m_raw * p.scale_log2;  // scale > 0
      if (j == 0) {
        m_used = m_blk;
      } else {
        float m_new = fmaxf(m_used, m_blk);
        bool need = m_new > m_used + 8.0f;
        if (__any_sync(0xffffffffu, need)) {
          // O may only be touched once PV(j-1) has landed
          mbar_wait(&pv_done[(j - 1) & 1], ((j - 1) >> 1) & 1);
          tc_fence_after();
          float alpha = need ? exp2f(m_used - m_new) : 1.0f;
#pragma unroll 1
          for (int c = 0; c < DPAD / 32; ++c) {
            uint32_t o[32];
            tmem_ld32(tmem + lane_addr + O_COL + c * 32, o);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
            tmem_st32(tmem + lane_addr + O_COL + c * 32, o);
          }
          tmem_st_wait();
          l *= alpha;
          if (need) m_used = m_new;
        }
      }
      float sm[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      const float neg_m = -m_used;
      // P buffer s was read by PV(j-2): waited for before the exponentials, so that they, the packs and the shared
      // stores are one basic block and interleave (see attention_split_kernel)
      if (j >= 2) mbar_wait(&pv_done[s], ((j - 2) >> 1) & 1);
#pragma unroll
      for (int c = 0; c < AKV; ++c) {
        t[c] = fast_exp2(fmaf(t[c], p.scale_log2, neg_m));
        sm[c & 7] += t[c];
      }
      l += ((sm[0] + sm[1]) + (sm[2] + sm[3])) + ((sm[4] + sm[5]) + (sm[6] + sm[7]));
      uint8_t* prow = p_s + s * P_BYTES + r * 128;
#pragma unroll
      for (int c16 = 0; c16 < 8; ++c16) {
        __half2 h0 = __floats2half2_rn(t[c16 * 8 + 0], t[c16 * 8 + 1]);
        __half2 h1 = __floats2half2_rn(t[c16 * 8 + 2], t[c16 * 8 + 3]);
        __half2 h2 = __floats2half2_rn(t[c16 * 8 + 4], t[c16 * 8 + 5]);
        __half2 h3 = __floats2half2_rn(t[c16 * 8 + 6], t[c16 * 8 + 7]);
        uint4 u;
        u.x = *reinterpret_cast<uint32_t*>(&h0);
        u.y = *reinterpret_cast<uint32_t*>(&h1);
        u.z = *reinterpret_cast<uint32_t*>(&h2);
        u.w = *reinterpret_cast<uint32_t*>(&h3);
        *reinterpret_cast<uint4*>(prow + ((c16 ^ (r & 7)) << 4)) = u;
      }
      fence_proxy_async();
      tc_fence_before();
      mbar_arrive(&p_full[s]);
    }
    // epilogue: O / l
    if (n_iter > 0) {
      mbar_wait(&pv_done[(n_iter - 1) & 1], ((n_iter - 1) >> 1) & 1);
      tc_fence_after();
    }
    const float inv_l = l > 0.f ? 1.0f / l : 0.f;
    __half* orow = p.out + static_cast<size_t>(b) * p.o_batch_stride + static_cast<size_t>(qi) * p.ldo + head * p.d;
#pragma unroll 1
    for (int c = 0; c < DPAD / 32; ++c) {
      if (c * 32 >= p.d) break;
      uint32_t o[32];
      tmem_ld32(tmem + lane_addr + O_COL + c * 32, o);
      tmem_ld_wait();
      if (qi < p.nq && n_iter > 0) {
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          int col = c * 32 + i;
          if (col < p.d)
            *reinterpret_cast<__half2*>(orow + col) =
                __floats2half2_rn(__uint_as_float(o[i]) * inv_l, __uint_as_float(o[i + 1]) * inv_l);
        }
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, TMEM_COLS);
  }
}


// ---------------------------------------------------------------------------------------------------------------------
// Split-state variant for DPAD == 64, d < 64 (the 64x64-latent self-attention of SD v1: N = 4096, d = 40 - 13 % of a
// UNet evaluation with the kernel above, which keeps one softmax thread per query row: 2 softmax warps per scheduler,
// MUFU pipe 42 % busy, the row maximum / exponent / pack phases of a warp strictly serial).
//
//   * every query row is handled by TWO threads, each owning 32 of the 64 key columns of a KV tile and its OWN online-
//     softmax state (running maximum) and its own output accumulator: O_A += P[:, 0:32] V[0:32], O_B += P[:, 32:64] V[32:64]
//     (the same four K = 16 MMAs, two per accumulator). The two halves never talk inside the loop; they are merged once
//     at the end: O = (2^(mA-m) O_A + 2^(mB-m) O_B) / (2^(mA-m) lA + 2^(mB-m) lB). Eight softmax warps per CTA, four per
//     scheduler with two co-resident CTAs, ~70 registers per thread.
//   * the row sums come out of the tensor cores: row d of every V^T tile in shared memory is a constant row of ones
//     (TMA only writes rows 0 .. d-1 of the tile; rows d .. 63 are initialised once), so column d of each accumulator
//     is sum_j P[i, j] - consistent with the fp16-rounded P the numerator uses, rescaled together with O, no FADD chain.
//   * the block maximum uses 3-input FMNMX.
constexpr int SPLIT_THREADS = 64 + 256;
constexpr int SPLIT_ST = 3;
constexpr int SPLIT_SMEM = AQ * 64 * 2 + SPLIT_ST * (2 * AKV * 64 * 2) + 2 * AQ * AKV * 2 + 1024;

__global__ void __launch_bounds__(SPLIT_THREADS, 2)
    attention_split_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                           const __grid_constant__ CUtensorMap tmV, const AttnArgs p) {
  constexpr int DPAD = 64;
  constexpr int Q_BYTES = AQ * DPAD * 2;
  constexpr int K_BYTES = AKV * DPAD * 2;
  constexpr int V_BYTES = DPAD * AKV * 2;
  constexpr int P_BYTES = AQ * AKV * 2;
  constexpr int TMEM_COLS = 256;
  constexpr int ST = SPLIT_ST;
  constexpr uint32_t O_COL = 128;   // O_A at 128, O_B at 192

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* q_s = smem;
  uint8_t* k_s = q_s + Q_BYTES;
  uint8_t* v_s = k_s + ST * K_BYTES;
  uint8_t* p_s = v_s + ST * V_BYTES;

  __shared__ uint64_t q_full, k_full[ST], v_full[ST], kv_empty[ST], s_full[2], p_full[2], pv_done[2];
  __shared__ uint32_t tmem_base_smem;
  __shared__ float m_sh[2][AQ];

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  pdl_launch_dependents();
  const int q0 = blockIdx.x * AQ;
  const int head = blockIdx.y;
  const int b = blockIdx.z;
  int nkv_eff = p.nkv;
  if (p.causal) nkv_eff = min(p.nkv, q0 + AQ);
  const int n_iter = (nkv_eff + AKV - 1) / AKV;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    mbar_init(&q_full, 1);
    for (int i = 0; i < ST; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&v_full[i], 1);
      mbar_init(&kv_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&p_full[i], 256);
      mbar_init(&pv_done[i], 1);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(&tmem_base_smem, TMEM_COLS);
    tmem_relinquish();
  }
  {
    // constant rows of the V^T tiles: row d = ones, rows d+1 .. 63 = zeros (16-byte granules; a constant row is
    // invariant under the 128-byte swizzle). TMA never writes them.
    const int granules = (DPAD - p.d) * 8;
    for (int i = threadIdx.x; i < ST * granules; i += SPLIT_THREADS) {
      const int st = i / granules, g = i - st * granules;
      const uint32_t val = (g < 8) ? 0x3C003C00u : 0u;
      *reinterpret_cast<uint4*>(v_s + st * V_BYTES + p.d * 128 + g * 16) = make_uint4(val, val, val, val);
    }
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_smem;

  pdl_wait();
  if (warp == 0) {
    if (elect_one()) {
      const uint32_t v_load_bytes = static_cast<uint32_t>(p.d) * AKV * 2;
      mbar_arrive_expect_tx(&q_full, Q_BYTES);
      tma_load_3d(q_s, &tmQ, &q_full, head * DPAD, q0, b);
      for (int j = 0; j < n_iter; ++j) {
        int s = j % ST;
        uint32_t ph = (j / ST) & 1;
        mbar_wait(&kv_empty[s], ph ^ 1);
        mbar_arrive_expect_tx(&k_full[s], K_BYTES);
        tma_load_3d(k_s + s * K_BYTES, &tmK, &k_full[s], head * DPAD, j * AKV, b);
        mbar_arrive_expect_tx(&v_full[s], v_load_bytes);
        tma_load_3d(v_s + s * V_BYTES, &tmV, &v_full[s], j * AKV, head * DPAD, b);
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc_s = umma_idesc_f16(AQ, AKV);
      // d < 64: only the K steps holding real Q / K columns are issued, and the two output accumulators are
      // ceil16(d + 1) columns wide (d value columns + the row-sum column d): d = 40 -> 3 of 4 K steps, N = 48 of 64
      const int ksteps = (p.d + 15) >> 4;
      const uint32_t idesc_o = umma_idesc_f16(AQ, min(DPAD, ((p.d + 16) >> 4) << 4));
      const uint32_t q_addr = smem_u32(q_s);
      auto issue_s = [&](int j) {
        const int s = j & 1;
        const int ks = j % ST;
        mbar_wait(&k_full[ks], (j / ST) & 1);
        tc_fence_after();
        const uint32_t k_addr = smem_u32(k_s + ks * K_BYTES);
#pragma unroll
        for (int kk = 0; kk < DPAD / 16; ++kk) {
          if (kk >= ksteps) break;
          uint64_t da = umma_desc_k128(q_addr + kk * 32);
          uint64_t db = umma_desc_k128(k_addr + kk * 32);
          umma_f16(tmem + s * AKV, da, db, idesc_s, kk > 0 ? 1u : 0u);
        }
        umma_commit(&s_full[s]);
      };
      mbar_wait(&q_full, 0);
      if (n_iter > 0) issue_s(0);
      for (int j = 0; j < n_iter; ++j) {
        int s = j & 1;
        uint32_t ph = (j >> 1) & 1;
        if (j + 1 < n_iter) issue_s(j + 1);
        const int ks = j % ST;
        mbar_wait(&p_full[s], ph);
        mbar_wait(&v_full[ks], (j / ST) & 1);
        tc_fence_after();
        const uint32_t p_addr = smem_u32(p_s + s * P_BYTES);
        const uint32_t v_addr = smem_u32(v_s + ks * V_BYTES);
#pragma unroll
        for (int kk = 0; kk < AKV / 16; ++kk) {   // key columns 0-31 -> O_A, 32-63 -> O_B
          uint64_t da = umma_desc_k128(p_addr + kk * 32);
          uint64_t db = umma_desc_k128(v_addr + kk * 32);
          umma_f16(tmem + O_COL + (kk >> 1) * DPAD, da, db, idesc_o, (j > 0 || (kk & 1)) ? 1u : 0u);
        }
        umma_commit(&kv_empty[ks]);
        umma_commit(&pv_done[s]);
      }
    }
  } else {
    const int lg = warp & 3;
    const int hf = (warp - 2) >> 2;   // key-column half of every KV tile this thread owns
    const int r = lg * 32 + lane;
    const int qi = q0 + r;
    const uint32_t lane_addr = static_cast<uint32_t>(lg * 32) << 16;
    const uint32_t o_addr = tmem + lane_addr + O_COL + hf * DPAD;
    float m_used = -INFINITY;
    for (int j = 0; j < n_iter; ++j) {
      const int s = j & 1;
      mbar_wait(&s_full[s], (j >> 1) & 1);
      tc_fence_after();
      float t[32];
      {
        uint32_t r0[32];
        tmem_ld32(tmem + lane_addr + s * AKV + hf * 32, r0);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < 32; ++c) t[c] = __uint_as_float(r0[c]);
      }
      const int kv0 = j * AKV + hf * 32;
      if ((kv0 + 32 > p.nkv) || (p.causal && kv0 + 31 > q0)) {
#pragma unroll
        for (int c = 0; c < 32; ++c) {
          int kv = kv0 + c;
          if ((kv >= p.nkv) || (p.causal && kv > qi)) t[c] = -INFINITY;
        }
      }
      float mx[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) mx[i] = fmaxf(fmaxf(t[i], t[4 + i]), t[8 + i]);
#pragma unroll
      for (int i = 0; i < 4; ++i) mx[i] = fmaxf(fmaxf(mx[i], t[12 + i]), t[16 + i]);
#pragma unroll
      for (int i = 0; i < 4; ++i) mx[i] = fmaxf(fmaxf(mx[i], t[20 + i]), t[24 + i]);
#pragma unroll
      for (int i = 0; i < 4; ++i) mx[i] = fmaxf(mx[i], t[28 + i]);
      const float m_blk = fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3])) * p.scale_log2;  // scale > 0
      {
        const float m_new = fmaxf(m_used, m_blk);
        const bool need = m_new > m_used + 8.0f;   // also true for the first finite block (m_used = -inf)
        if (j > 0 && __any_sync(0xffffffffu, need)) {
          mbar_wait(&pv_done[(j - 1) & 1], ((j - 1) >> 1) & 1);   // O may only be touched once PV(j-1) has landed
          tc_fence_after();
          const float alpha = need ? exp2f(m_used - m_new) : 1.0f;   // exp2f(-inf) = 0: nothing accumulated yet
#pragma unroll 1
          for (int c = 0; c < DPAD / 32; ++c) {
            uint32_t o[32];
            tmem_ld32(o_addr + c * 32, o);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
            tmem_st32(o_addr + c * 32, o);
          }
          tmem_st_wait();
        }
        if (need) m_used = m_new;
      }
      const float neg_m = (m_used == -INFINITY) ? 0.f : -m_used;   // a fully masked half so far: exp2(-inf) = 0
      // P buffer s was read by PV(j-2). Waited for BEFORE the exponentials (it completed long ago) so that scale /
      // exponent / pack / store form one basic block: the packs and shared stores then issue between the MUFU
      // instructions instead of after them (all softmax warps of an SM reach the MUFU phase together; whatever issues
      // inside that phase is free)
      if (j >= 2) mbar_wait(&pv_done[s], ((j - 2) >> 1) & 1);
#pragma unroll
      for (int c = 0; c < 32; ++c) t[c] = fast_exp2(fmaf(t[c], p.scale_log2, neg_m));
      uint8_t* prow = p_s + s * P_BYTES + r * 128;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        __half2 h0 = __floats2half2_rn(t[i * 8 + 0], t[i * 8 + 1]);
        __half2 h1 = __floats2half2_rn(t[i * 8 + 2], t[i * 8 + 3]);
        __half2 h2 = __floats2half2_rn(t[i * 8 + 4], t[i * 8 + 5]);
        __half2 h3 = __floats2half2_rn(t[i * 8 + 6], t[i * 8 + 7]);
        uint4 u;
        u.x = *reinterpret_cast<uint32_t*>(&h0);
        u.y = *reinterpret_cast<uint32_t*>(&h1);
        u.z = *reinterpret_cast<uint32_t*>(&h2);
        u.w = *reinterpret_cast<uint32_t*>(&h3);
        *reinterpret_cast<uint4*>(prow + (((hf * 4 + i) ^ (r & 7)) << 4)) = u;
      }
      fence_proxy_async();
      tc_fence_before();
      mbar_arrive(&p_full[s]);
    }
    // merge the two halves: O = (fA O_A + fB O_B) / (fA lA + fB lB), l = column d of each accumulator
    m_sh[hf][r] = m_used;
    asm volatile("bar.sync 1, 256;" ::: "memory");
    if (n_iter > 0) {
      mbar_wait(&pv_done[(n_iter - 1) & 1], ((n_iter - 1) >> 1) & 1);
      tc_fence_after();
    }
    const float mA = m_sh[0][r], mB = m_sh[1][r];
    const float m = fmaxf(mA, mB);
    const float fA = (mA == -INFINITY) ? 0.f : exp2f(mA - m);
    const float fB = (mB == -INFINITY) ? 0.f : exp2f(mB - m);
    const uint32_t oa = tmem + lane_addr + O_COL, ob = oa + DPAD;
    float inv_l = 0.f;
    uint32_t a[32], bb[32];
    if (n_iter > 0) {
      const uint32_t la = tmem_ld1(oa + p.d), lb = tmem_ld1(ob + p.d);
      tmem_ld32(oa + hf * 32, a);
      tmem_ld32(ob + hf * 32, bb);
      tmem_ld_wait();
      const float l = fA * __uint_as_float(la) + fB * __uint_as_float(lb);
      inv_l = l > 0.f ? 1.0f / l : 0.f;
    }
    if (qi < p.nq && n_iter > 0) {
      __half* orow = p.out + static_cast<size_t>(b) * p.o_batch_stride + static_cast<size_t>(qi) * p.ldo + head * p.d;
      const float ga = fA * inv_l, gb = fB * inv_l;
#pragma unroll
      for (int i = 0; i < 32; i += 2) {
        const int col = hf * 32 + i;
        if (col < p.d)
          *reinterpret_cast<__half2*>(orow + col) =
              __floats2half2_rn(__uint_as_float(a[i]) * ga + __uint_as_float(bb[i]) * gb,
                                __uint_as_float(a[i + 1]) * ga + __uint_as_float(bb[i + 1]) * gb);
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, TMEM_COLS);
  }
}


// ---------------------------------------------------------------------------------------------------------------------
// Wide single-head variant: d = 512 (the AutoencoderKL mid-block AttnBlock, ldm/modules/diffusionmodules/model.py:178-202:
// softmax(q k^T / sqrt(c)) v over h*w tokens with c = 512 channels). The reference - and the first version of this
// engine - materialise the N x N logits (64 MiB fp32 per 512^2 image, 324 MiB at 768^2); here they never leave the SM:
//   * one CTA = 128 query rows x ONE 256-column slice of the output (grid.y = 2 slices; S is recomputed per slice:
//     the accumulator O of a 512-wide head does not fit the 512 TMEM columns next to S);
//   * Q (128 x 512 fp16 = 128 KB) stays resident in shared memory as eight 64-column panels; K streams through a ring of
//     64 x 64 panels, S(j) = sum over the eight panels (32 MMAs, K = 16 each) into a double-buffered TMEM tile;
//   * V^T slice tiles [256 x 64] and the fp16 P tile are single-buffered (shared memory is full), released by PV(j-1);
//   * softmax / lazy rescale / epilogue as in attention_tc_kernel (one query row per thread).
constexpr int WIDE_D = 512;
constexpr int WIDE_DV = 256;
constexpr int WIDE_KST = 4;                      // K panel ring depth
constexpr int WIDE_PANELS = WIDE_D / 64;
constexpr int WIDE_SMEM = AQ * WIDE_D * 2 + WIDE_KST * (AKV * 64 * 2) + WIDE_DV * AKV * 2 + AQ * AKV * 2 + 1024;

__global__ void __launch_bounds__(192, 1)
    attention_wide_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                          const __grid_constant__ CUtensorMap tmV, const AttnArgs p) {
  constexpr int Q_BYTES = AQ * WIDE_D * 2;
  constexpr int KP_BYTES = AKV * 64 * 2;          // one K panel
  constexpr int V_BYTES = WIDE_DV * AKV * 2;
  constexpr int TMEM_COLS = 512;
  constexpr uint32_t O_COL = 128;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* q_s = smem;
  uint8_t* k_s = q_s + Q_BYTES;
  uint8_t* v_s = k_s + WIDE_KST * KP_BYTES;
  uint8_t* p_s = v_s + V_BYTES;

  __shared__ uint64_t q_full, k_full[WIDE_KST], k_empty[WIDE_KST], v_full, s_full[2], p_full, pv_done;
  __shared__ uint32_t tmem_base_smem;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  pdl_launch_dependents();
  const int q0 = blockIdx.x * AQ;
  const int dv0 = blockIdx.y * WIDE_DV;
  const int b = blockIdx.z;
  const int n_iter = (p.nkv + AKV - 1) / AKV;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    mbar_init(&q_full, 1);
    for (int i = 0; i < WIDE_KST; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&k_empty[i], 1);
    }
    mbar_init(&v_full, 1);
    mbar_init(&s_full[0], 1);
    mbar_init(&s_full[1], 1);
    mbar_init(&p_full, 128);
    mbar_init(&pv_done, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(&tmem_base_smem, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_smem;

  pdl_wait();
  if (warp == 0) {
    if (elect_one()) {
      mbar_arrive_expect_tx(&q_full, Q_BYTES);
      for (int pn = 0; pn < WIDE_PANELS; ++pn) tma_load_3d(q_s + pn * (AQ * 128), &tmQ, &q_full, pn * 64, q0, b);
      int ks = 0;
      uint32_t kph = 0;
      for (int j = 0; j < n_iter; ++j) {
        for (int pn = 0; pn < WIDE_PANELS; ++pn) {
          mbar_wait(&k_empty[ks], kph ^ 1);
          mbar_arrive_expect_tx(&k_full[ks], KP_BYTES);
          tma_load_3d(k_s + ks * KP_BYTES, &tmK, &k_full[ks], pn * 64, j * AKV, b);
          if (++ks == WIDE_KST) {
            ks = 0;
            kph ^= 1;
          }
        }
        if (j > 0) mbar_wait(&pv_done, (j - 1) & 1);   // PV(j-1) has read the single V^T buffer
        mbar_arrive_expect_tx(&v_full, V_BYTES);
        tma_load_3d(v_s, &tmV, &v_full, j * AKV, dv0, b);
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc_s = umma_idesc_f16(AQ, AKV);
      constexpr uint32_t idesc_o = umma_idesc_f16(AQ, WIDE_DV);
      const uint32_t q_addr = smem_u32(q_s);
      int ks = 0;
      uint32_t kph = 0;
      auto issue_s = [&](int j) {
        const int s = j & 1;
        for (int pn = 0; pn < WIDE_PANELS; ++pn) {
          mbar_wait(&k_full[ks], kph);
          tc_fence_after();
          const uint32_t k_addr = smem_u32(k_s + ks * KP_BYTES);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
            uint64_t da = umma_desc_k128(q_addr + pn * (AQ * 128) + kk * 32);
            uint64_t db = umma_desc_k128(k_addr + kk * 32);
            umma_f16(tmem + s * AKV, da, db, idesc_s, (pn > 0 || kk > 0) ? 1u : 0u);
          }
          umma_commit(&k_empty[ks]);
          if (++ks == WIDE_KST) {
            ks = 0;
            kph ^= 1;
          }
        }
        umma_commit(&s_full[s]);
      };
      mbar_wait(&q_full, 0);
      if (n_iter > 0) issue_s(0);
      for (int j = 0; j < n_iter; ++j) {
        if (j + 1 < n_iter) issue_s(j + 1);
        mbar_wait(&p_full, j & 1);
        mbar_wait(&v_full, j & 1);
        tc_fence_after();
        const uint32_t p_addr = smem_u32(p_s);
        const uint32_t v_addr = smem_u32(v_s);
#pragma unroll
        for (int kk = 0; kk < AKV / 16; ++kk) {
          uint64_t da = umma_desc_k128(p_addr + kk * 32);
          uint64_t db = umma_desc_k128(v_addr + kk * 32);
          umma_f16(tmem + O_COL, da, db, idesc_o, (j > 0 || kk > 0) ? 1u : 0u);
        }
        umma_commit(&pv_done);
      }
    }
  } else {
    const int lg = warp & 3;
    const int r = lg * 32 + lane;
    const int qi = q0 + r;
    const uint32_t lane_addr = static_cast<uint32_t>(lg * 32) << 16;
    float m_used = -INFINITY;
    float l = 0.f;
    for (int j = 0; j < n_iter; ++j) {
      const int s = j & 1;
      mbar_wait(&s_full[s], (j >> 1) & 1);
      tc_fence_after();
      float t[AKV];
      {
        uint32_t r0[32], r1[32];
        tmem_ld32(tmem + lane_addr + s * AKV, r0);
        tmem_ld32(tmem + lane_addr + s * AKV + 32, r1);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < 32; ++c) {
          t[c] = __uint_as_float(r0[c]);
          t[32 + c] = __uint_as_float(r1[c]);
        }
      }
      const int kv0 = j * AKV;
      if (kv0 + AKV > p.nkv) {
#pragma unroll
        for (int c = 0; c < AKV; ++c)
          if (kv0 + c >= p.nkv) t[c] = -INFINITY;
      }
      float mx[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) mx[i] = t[i];
#pragma unroll
      for (int c = 8; c < AKV; ++c) mx[c & 7] = fmaxf(mx[c & 7], t[c]);
      const float m_blk =
          fmaxf(fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3])), fmaxf(fmaxf(mx[4], mx[5]), fmaxf(mx[6], mx[7]))) * p.scale_log2;
      if (j == 0) {
        m_used = m_blk;
      } else {
        // the single P / V buffers: PV(j-1) must have finished before P(j) is written anyway, so wait for it here and
        // rescale O directly when the running maximum moved
        mbar_wait(&pv_done, (j - 1) & 1);
        tc_fence_after();
        const float m_new = fmaxf(m_used, m_blk);
        const bool need = m_new > m_used + 8.0f;
        if (__any_sync(0xffffffffu, need)) {
          const float alpha = need ? exp2f(m_used - m_new) : 1.0f;
#pragma unroll 1
          for (int c = 0; c < WIDE_DV / 32; ++c) {
            uint32_t o[32];
            tmem_ld32(tmem + lane_addr + O_COL + c * 32, o);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
            tmem_st32(tmem + lane_addr + O_COL + c * 32, o);
          }
          tmem_st_wait();
          l *= alpha;
          if (need) m_used = m_new;
        }
      }
      float sm[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      const float neg_m = -m_used;
#pragma unroll
      for (int c = 0; c < AKV; ++c) {
        t[c] = fast_exp2(fmaf(t[c], p.scale_log2, neg_m));
        sm[c & 7] += t[c];
      }
      l += ((sm[0] + sm[1]) + (sm[2] + sm[3])) + ((sm[4] + sm[5]) + (sm[6] + sm[7]));
      uint8_t* prow = p_s + r * 128;
#pragma unroll
      for (int c16 = 0; c16 < 8; ++c16) {
        __half2 h0 = __floats2half2_rn(t[c16 * 8 + 0], t[c16 * 8 + 1]);
        __half2 h1 = __floats2half2_rn(t[c16 * 8 + 2], t[c16 * 8 + 3]);
        __half2 h2 = __floats2half2_rn(t[c16 * 8 + 4], t[c16 * 8 + 5]);
        __half2 h3 = __floats2half2_rn(t[c16 * 8 + 6], t[c16 * 8 + 7]);
        uint4 u;
        u.x = *reinterpret_cast<uint32_t*>(&h0);
        u.y = *reinterpret_cast<uint32_t*>(&h1);
        u.z = *reinterpret_cast<uint32_t*>(&h2);
        u.w = *reinterpret_cast<uint32_t*>(&h3);
        *reinterpret_cast<uint4*>(prow + ((c16 ^ (r & 7)) << 4)) = u;
      }
      fence_proxy_async();
      tc_fence_before();
      mbar_arrive(&p_full);
    }
    if (n_iter > 0) {
      mbar_wait(&pv_done, (n_iter - 1) & 1);
      tc_fence_after();
    }
    const float inv_l = l > 0.f ? 1.0f / l : 0.f;
    __half* orow = p.out + static_cast<size_t>(b) * p.o_batch_stride + static_cast<size_t>(qi) * p.ldo + dv0;
#pragma unroll 1
    for (int c = 0; c < WIDE_DV / 32; ++c) {
      uint32_t o[32];
      tmem_ld32(tmem + lane_addr + O_COL + c * 32, o);
      tmem_ld_wait();
      if (qi < p.nq && n_iter > 0) {
#pragma unroll
        for (int i = 0; i < 32; i += 8) {
          __half2 h0 = __floats2half2_rn(__uint_as_float(o[i]) * inv_l, __uint_as_float(o[i + 1]) * inv_l);
          __half2 h1 = __floats2half2_rn(__uint_as_float(o[i + 2]) * inv_l, __uint_as_float(o[i + 3]) * inv_l);
          __half2 h2 = __floats2half2_rn(__uint_as_float(o[i + 4]) * inv_l, __uint_as_float(o[i + 5]) * inv_l);
          __half2 h3 = __floats2half2_rn(__uint_as_float(o[i + 6]) * inv_l, __uint_as_float(o[i + 7]) * inv_l);
          uint4 u;
          u.x = *reinterpret_cast<uint32_t*>(&h0);
          u.y = *reinterpret_cast<uint32_t*>(&h1);
          u.z = *reinterpret_cast<uint32_t*>(&h2);
          u.w = *reinterpret_cast<uint32_t*>(&h3);
          *reinterpret_cast<uint4*>(orow + c * 32 + i) = u;
        }
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, TMEM_COLS);
  }
}

template <int DPAD>
static int launch_attn(const CUtensorMap& q, const CUtensorMap& k, const CUtensorMap& v, const AttnArgs& p, dim3 grid,
                       cudaStream_t st) {
  constexpr int SMEM = AttnCfg<DPAD>::SMEM;
  auto kern = attention_tc_kernel<DPAD>;
  static bool configured = false;
  if (!configured) {
    SDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    configured = true;
  }
  SDB_CUDA(launch_pdl(kern, grid, dim3(192), SMEM, st, q, k, v, p));
  SDB_LAUNCH_CHECK();
  return 0;
}

}  // namespace sdb

using namespace sdb;

extern "C" int sdb_attention(const sdb_attn_desc* d, sdb_stream_t stream) {
  if (d && ::sdb::plan_recording()) {
    const sdb_attn_desc c = *d;
    ::sdb::plan_record([c](cudaStream_t s_) { return sdb_attention(&c, s_); });
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SDB_CHECK(d && d->q && d->k && d->vt && d->out, "sdb_attention: null pointer");
  if (d->dpad == WIDE_D) {
    // single-head d = 512 (AutoencoderKL AttnBlock): q, k [B, n, 512], vt [B, 512, ldvt]
    SDB_CHECK(d->d == WIDE_D && d->heads == 1 && !d->causal, "sdb_attention: dpad 512 is the single-head d = 512 kernel");
    SDB_CHECK(d->batch > 0 && d->nq > 0 && d->nkv > 0, "sdb_attention: bad sizes");
    SDB_CHECK(d->ldq % 8 == 0 && d->ldk % 8 == 0 && d->ldvt % 8 == 0 && d->ldo % 8 == 0 && d->o_batch_stride % 8 == 0,
              "sdb_attention: leading dims must be multiples of 8");
    CUtensorMap tq, tk, tv;
    {
      uint64_t dims[3] = {WIDE_D, static_cast<uint64_t>(d->nq), static_cast<uint64_t>(d->batch)};
      uint64_t str[2] = {static_cast<uint64_t>(d->ldq) * 2, static_cast<uint64_t>(d->q_batch_stride) * 2};
      uint32_t box[3] = {64, AQ, 1};
      if (make_tmap_f16(&tq, d->q, 3, dims, str, box)) return 1;
    }
    {
      uint64_t dims[3] = {WIDE_D, static_cast<uint64_t>(d->nkv), static_cast<uint64_t>(d->batch)};
      uint64_t str[2] = {static_cast<uint64_t>(d->ldk) * 2, static_cast<uint64_t>(d->k_batch_stride) * 2};
      uint32_t box[3] = {64, AKV, 1};
      if (make_tmap_f16(&tk, d->k, 3, dims, str, box)) return 1;
    }
    {
      uint64_t dims[3] = {static_cast<uint64_t>(d->nkv), WIDE_D, static_cast<uint64_t>(d->batch)};
      uint64_t str[2] = {static_cast<uint64_t>(d->ldvt) * 2, static_cast<uint64_t>(d->vt_batch_stride) * 2};
      uint32_t box[3] = {AKV, WIDE_DV, 1};
      if (make_tmap_f16(&tv, d->vt, 3, dims, str, box)) return 1;
    }
    AttnArgs p{};
    p.nq = d->nq;
    p.nkv = d->nkv;
    p.d = d->d;
    p.heads = 1;
    p.ldo = d->ldo;
    p.o_batch_stride = d->o_batch_stride;
    p.out = static_cast<__half*>(d->out);
    p.scale_log2 = d->scale * 1.4426950408889634f;
    p.causal = 0;
    static bool configured = false;
    if (!configured) {
      SDB_CUDA(cudaFuncSetAttribute(attention_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, WIDE_SMEM));
      configured = true;
    }
    dim3 grid((d->nq + AQ - 1) / AQ, WIDE_D / WIDE_DV, d->batch);
    SDB_CUDA(launch_pdl(attention_wide_kernel, grid, dim3(192), WIDE_SMEM, st, tq, tk, tv, p));
    SDB_LAUNCH_CHECK();
    return 0;
  }
  SDB_CHECK(d->dpad == 64 || d->dpad == 128 || d->dpad == 192, "sdb_attention: dpad must be 64/128/192/512 (got %d)",
            d->dpad);
  SDB_CHECK(d->d > 0 && d->d <= d->dpad && d->d % 2 == 0, "sdb_attention: bad head dim %d", d->d);
  SDB_CHECK(d->batch > 0 && d->heads > 0 && d->nq > 0 && d->nkv > 0, "sdb_attention: bad sizes");
  SDB_CHECK(d->ldq % 8 == 0 && d->ldk % 8 == 0 && d->ldvt % 8 == 0, "sdb_attention: leading dims must be multiples of 8");
  SDB_CHECK(d->ldo % 2 == 0 && d->o_batch_stride % 2 == 0, "sdb_attention: output stride must be even");

  CUtensorMap tq, tk, tv;
  const uint64_t hd = static_cast<uint64_t>(d->heads) * d->dpad;
  {
    uint64_t dims[3] = {hd, static_cast<uint64_t>(d->nq), static_cast<uint64_t>(d->batch)};
    uint64_t str[2] = {static_cast<uint64_t>(d->ldq) * 2, static_cast<uint64_t>(d->q_batch_stride) * 2};
    uint32_t box[3] = {64, AQ, 1};
    if (make_tmap_f16(&tq, d->q, 3, dims, str, box)) return 1;
  }
  {
    uint64_t dims[3] = {hd, static_cast<uint64_t>(d->nkv), static_cast<uint64_t>(d->batch)};
    uint64_t str[2] = {static_cast<uint64_t>(d->ldk) * 2, static_cast<uint64_t>(d->k_batch_stride) * 2};
    uint32_t box[3] = {64, AKV, 1};
    if (make_tmap_f16(&tk, d->k, 3, dims, str, box)) return 1;
  }
  // split-state kernel (two threads per query row, row sums from a ones row of V^T): dpad 64 with spare rows
  const bool use_split = d->dpad == 64 && d->d < 64 && d->d % 8 == 0;
  {
    uint64_t dims[3] = {static_cast<uint64_t>(d->nkv), hd, static_cast<uint64_t>(d->batch)};
    uint64_t str[2] = {static_cast<uint64_t>(d->ldvt) * 2, static_cast<uint64_t>(d->vt_batch_stride) * 2};
    uint32_t box[3] = {AKV, static_cast<uint32_t>(use_split ? d->d : d->dpad), 1};   // split: only the d real rows
    if (make_tmap_f16(&tv, d->vt, 3, dims, str, box)) return 1;
  }
  AttnArgs p{};
  p.nq = d->nq;
  p.nkv = d->nkv;
  p.d = d->d;
  p.heads = d->heads;
  p.ldo = d->ldo;
  p.o_batch_stride = d->o_batch_stride;
  p.out = static_cast<__half*>(d->out);
  p.scale_log2 = d->scale * 1.4426950408889634f;
  p.causal = d->causal;
  dim3 grid((d->nq + AQ - 1) / AQ, d->heads, d->batch);
  if (use_split) {
    static bool configured = false;
    if (!configured) {
      SDB_CUDA(cudaFuncSetAttribute(attention_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SPLIT_SMEM));
      configured = true;
    }
    SDB_CUDA(launch_pdl(attention_split_kernel, grid, dim3(SPLIT_THREADS), SPLIT_SMEM, st, tq, tk, tv, p));
    SDB_LAUNCH_CHECK();
    return 0;
  }
  switch (d->dpad) {
    case 64: return launch_attn<64>(tq, tk, tv, p, grid, st);
    case 128: return launch_attn<128>(tq, tk, tv, p, grid, st);
    default: return launch_attn<192>(tq, tk, tv, p, grid, st);
  }
}
