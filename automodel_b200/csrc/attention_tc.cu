// Causal GQA flash attention on the 5th-gen tensor cores (tcgen05.mma, TMEM accumulators, TMA loads), sm_100a.
// Same contract as attention.cu (token-major q/k/v views, cu_seqlens, lse [Hq,T]); see that file for the reference
// call sites.  Forward:
//   CTA = one 128-row q tile of one (sequence, head); loops over 128-row kv tiles up to the diagonal.
//   warp 0      TMA producer: Q once, K/V tiles through 2-stage rings (128B-swizzled boxes of 64 columns)
//   warp 1      MMA issuer (one thread): S_j = Q K_j^T into one of two TMEM S buffers (so S_{j+1} overlaps softmax_j),
//               O += P_j V_j (A = P from smem, K-major; B = V, MN-major descriptor - no transpose of V anywhere)
//   warps 2..5  softmax: each thread owns ONE q row (= TMEM lane): row max / sum need no shuffles.  S row -> registers
//               (tcgen05.ld), online softmax with lazy rescaling (O in TMEM is only touched when the running max grows
//               by more than 2^8), P -> bf16 -> swizzled smem, final O / l -> global.
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <math.h>
#include <stdio.h>

#include "common.h"
#include "ptx.cuh"

namespace b200 {

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <int D>
struct AttnFwdSmem {
  static constexpr int TILE = 128 * D * 2;       // one Q/K/V tile: D/64 boxes of [128 rows x 64 cols]
  static constexpr int P_BYTES = 128 * 128 * 2;  // two K-major atoms of 64 kv columns
  static constexpr int Q_OFF = 0;
  static constexpr int K_OFF = TILE;
  static constexpr int V_OFF = 3 * TILE;
  static constexpr int P_OFF = 5 * TILE;
  static constexpr int XCH_OFF = P_OFF + P_BYTES;        // float [2][2][128] running-max exchange + [2][128] row-sum exchange
  static constexpr int BAR_OFF = XCH_OFF + 768 * 4;
  static constexpr int NUM_BARS = 1 + 4 + 4 + 2 + 2 + 1 + 1;  // q_full, k_full/empty[2], v_full/empty[2], s_full[2], s_free[2], p_ready, pv_done
  static constexpr int DYN = BAR_OFF + NUM_BARS * 8 + 16 + 1024;
};

template <int D>
__global__ void __launch_bounds__(320, 1)
attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                   const __grid_constant__ CUtensorMap tmV, __nv_bfloat16* __restrict__ o, float* __restrict__ lse,
                   const int* __restrict__ cu_seqlens, int64_t ldo, int Hq, int Hkv, int T, float scale_log2) {
  using L = AttnFwdSmem<D>;
  constexpr int ATOMS = D / 64;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);
  uint64_t* q_full = bars;
  uint64_t* k_full = bars + 1;
  uint64_t* k_empty = bars + 3;
  uint64_t* v_full = bars + 5;
  uint64_t* v_empty = bars + 7;
  uint64_t* s_full = bars + 9;
  uint64_t* s_free = bars + 11;
  uint64_t* p_ready = bars + 13;
  uint64_t* pv_done = bars + 14;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bars + L::NUM_BARS);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int seq = blockIdx.z, h = blockIdx.y;
  const int mt = gridDim.x - 1 - blockIdx.x;  // heavy tiles first
  const int s0 = cu_seqlens[seq];
  const int len = cu_seqlens[seq + 1] - s0;
  const int m0 = mt * 128;
  if (m0 >= len) return;  // uniform for the CTA, before any barrier / TMEM use
  const int hk = h / (Hq / Hkv);
  const int n_kv = min(mt + 1, (len + 127) / 128);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    mbar_init(q_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&k_empty[i], 1);
      mbar_init(&v_full[i], 1);
      mbar_init(&v_empty[i], 1);
      mbar_init(&s_full[i], 1);
      mbar_init(&s_free[i], 8);
    }
    mbar_init(p_ready, 8);
    mbar_init(pv_done, 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_holder, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;
  const uint32_t tS0 = tmem_base, tO = tmem_base + 256;

  if (warp == 0) {
    // ===================================================== TMA producer
    if (lane == 0) {
      mbar_arrive_expect_tx(q_full, L::TILE);
#pragma unroll
      for (int a = 0; a < ATOMS; ++a) tma_load_2d(smem + L::Q_OFF + a * 16384, &tmQ, q_full, h * D + a * 64, s0 + m0);
      for (int j = 0; j < n_kv; ++j) {
        const int st = j & 1;
        const uint32_t ph = ((j >> 1) & 1) ^ 1;
        mbar_wait(&k_empty[st], ph);
        mbar_arrive_expect_tx(&k_full[st], L::TILE);
#pragma unroll
        for (int a = 0; a < ATOMS; ++a)
          tma_load_2d(smem + L::K_OFF + st * L::TILE + a * 16384, &tmK, &k_full[st], hk * D + a * 64, s0 + j * 128);
        mbar_wait(&v_empty[st], ph);
        mbar_arrive_expect_tx(&v_full[st], L::TILE);
#pragma unroll
        for (int a = 0; a < ATOMS; ++a)
          tma_load_2d(smem + L::V_OFF + st * L::TILE + a * 16384, &tmV, &v_full[st], hk * D + a * 64, s0 + j * 128);
      }
    }
  } else if (warp == 1) {
    // ===================================================== MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc_s = make_idesc_bf16(128, 128, 0, 0);  // S = Q K^T : both K-major
      constexpr uint32_t idesc_o = make_idesc_bf16(128, D, 0, 1);    // O = P V   : A K-major, B (=V) MN-major
      const uint32_t q_base = smem_u32(smem + L::Q_OFF);
      const uint32_t p_base = smem_u32(smem + L::P_OFF);
      auto issue_s = [&](int j) {
        const int st = j & 1;
        mbar_wait(&k_full[st], (j >> 1) & 1);
        mbar_wait(&s_free[st], ((j >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t k_base = smem_u32(smem + L::K_OFF + st * L::TILE);
#pragma unroll
        for (int kk = 0; kk < D / 16; ++kk) {
          const uint32_t off = (kk >> 2) * 16384 + (kk & 3) * 32;
          umma_bf16(tS0 + st * 128, make_smem_desc_sw128(q_base + off, 16, 1024), make_smem_desc_sw128(k_base + off, 16, 1024),
                    idesc_s, kk != 0 ? 1u : 0u);
        }
        umma_commit(&k_empty[st]);
        umma_commit(&s_full[st]);
      };
      mbar_wait(q_full, 0);
      issue_s(0);
      for (int j = 0; j < n_kv; ++j) {
        if (j + 1 < n_kv) issue_s(j + 1);
        const int st = j & 1;
        mbar_wait(p_ready, j & 1);
        mbar_wait(&v_full[st], (j >> 1) & 1);
        tc_fence_after();
        const uint32_t v_base = smem_u32(smem + L::V_OFF + st * L::TILE);
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) {  // 128 kv rows / 16
          const uint64_t da = make_smem_desc_sw128(p_base + (kk >> 2) * 16384 + (kk & 3) * 32, 16, 1024);
          const uint64_t db = make_smem_desc_sw128(v_base + kk * 2048, 16384, 1024);
          umma_bf16(tO, da, db, idesc_o, (j | kk) != 0 ? 1u : 0u);
        }
        umma_commit(&v_empty[st]);
        umma_commit(pv_done);
      }
    }
  } else {
    // ===================================================== 8 softmax warps: thread <-> (q row r, half of the 128 kv columns).
    // Two warps per scheduler (instead of one) hide TMEM / MUFU latency; the two halves of a row agree on the running max through
    // shared memory (one named barrier per kv tile) and keep separate row sums that are combined once at the end.
    const int quad = warp & 3;                   // TMEM lane quarter this warp may access
    const int half = (warp - 2) >> 2;            // 0: kv columns [0,64), 1: [64,128)
    const int r = quad * 32 + lane;              // q row within the tile == TMEM lane
    const uint32_t lane_addr = static_cast<uint32_t>(quad * 32) << 16;
    const int qrow = m0 + r;                     // sequence-relative
    float m_used = 0.f, l_sum = 0.f;
    float* xch = reinterpret_cast<float*>(smem + L::XCH_OFF);  // [2 parity][2 halves][128 rows]
    uint8_t* p_row = smem + L::P_OFF + half * 16384 + r * 128;  // this half's K-major atom of P
    constexpr int OC = D / 64;                   // 32-column chunks of O owned by this half
    for (int j = 0; j < n_kv; ++j) {
      const int st = j & 1;
      mbar_wait(&s_full[st], (j >> 1) & 1);
      tc_fence_after();
      uint32_t v[2][32];
#pragma unroll
      for (int c = 0; c < 2; ++c) tmem_ld_32x32b_x32(tS0 + lane_addr + st * 128 + half * 64 + c * 32, v[c]);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_free[st]);  // S buffer may be overwritten by S_{j+2}

      const bool need_mask = (j == mt) || ((j + 1) * 128 > len);
      float mx = -INFINITY;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          float x = __uint_as_float(v[c][e]) * scale_log2;
          if (need_mask) {
            const int kv = j * 128 + half * 64 + c * 32 + e;
            if (kv > qrow || kv >= len) x = -INFINITY;
          }
          v[c][e] = __float_as_uint(x);
          mx = fmaxf(mx, x);
        }
      }
      // row max over both halves
      float* xc = xch + (j & 1) * 256;
      xc[half * 128 + r] = mx;
      asm volatile("bar.sync 1, 256;" ::: "memory");
      mx = fmaxf(mx, xc[(half ^ 1) * 128 + r]);
      if (j == 0) {
        m_used = (mx == -INFINITY) ? 0.f : mx;
      } else {
        // lazy rescale: only when the running max grew by more than 8 (P stays <= 2^8, exact in the final O / l).
        // Both halves of a row take the same decision (same mx, same m_used); each rescales its own half of the O columns.
        const bool grow = mx > m_used + 8.f;
        if (__any_sync(0xffffffffu, grow)) {
          mbar_wait(pv_done, (j - 1) & 1);  // O is quiescent: PV_{j-1} done, PV_j not yet issued
          tc_fence_after();
          const float f = grow ? ex2_approx(m_used - mx) : 1.f;
#pragma unroll
          for (int c = 0; c < OC; ++c) {
            uint32_t ov[32];
            tmem_ld_32x32b_x32(tO + lane_addr + (half * OC + c) * 32, ov);
            tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 32; ++e) ov[e] = __float_as_uint(__uint_as_float(ov[e]) * f);
            tmem_st_32x32b_x32(tO + lane_addr + (half * OC + c) * 32, ov);
          }
          tmem_st_wait();
          tc_fence_before();
          l_sum *= f;
          if (grow) m_used = mx;
        }
      }
      // P = 2^(x - m), partial row sum, bf16 pack
      uint32_t pk[32];
      float sum = 0.f;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
#pragma unroll
        for (int e = 0; e < 32; e += 2) {
          const float p0 = ex2_approx(__uint_as_float(v[c][e]) - m_used);
          const float p1 = ex2_approx(__uint_as_float(v[c][e + 1]) - m_used);
          sum += p0 + p1;
          pk[c * 16 + (e >> 1)] = pack_bf16x2(p0, p1);
        }
      }
      l_sum += sum;
      if (j > 0) mbar_wait(pv_done, (j - 1) & 1);  // P buffer free (PV_{j-1} has read it)
#pragma unroll
      for (int ch = 0; ch < 8; ++ch) {  // 8 chunks of 8 kv columns inside this half's atom
        uint4 val = make_uint4(pk[ch * 4], pk[ch * 4 + 1], pk[ch * 4 + 2], pk[ch * 4 + 3]);
        *reinterpret_cast<uint4*>(p_row + ((ch ^ (r & 7)) << 4)) = val;
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_ready);
    }
    // epilogue: combine the two half row sums, O / l -> bf16 -> global (each thread half a row of D elements)
    float* xl = xch + 512;  // [2 halves][128]
    xl[half * 128 + r] = l_sum;
    asm volatile("bar.sync 1, 256;" ::: "memory");
    l_sum += xl[(half ^ 1) * 128 + r];
    mbar_wait(pv_done, (n_kv - 1) & 1);
    tc_fence_after();
    const float inv = l_sum > 0.f ? 1.f / l_sum : 0.f;
    const bool valid = qrow < len;
    if (valid && half == 0) lse[static_cast<int64_t>(h) * T + s0 + qrow] = (m_used + log2f(l_sum)) * 0.6931471805599453f;
    __nv_bfloat16* orow = o + static_cast<int64_t>(s0 + qrow) * ldo + h * D + half * (D / 2);
#pragma unroll
    for (int c = 0; c < OC; ++c) {
      uint32_t ov[32];
      tmem_ld_32x32b_x32(tO + lane_addr + (half * OC + c) * 32, ov);
      tmem_ld_wait();
      if (valid) {
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {
          uint4 val;
          val.x = pack_bf16x2(__uint_as_float(ov[q4 * 8 + 0]) * inv, __uint_as_float(ov[q4 * 8 + 1]) * inv);
          val.y = pack_bf16x2(__uint_as_float(ov[q4 * 8 + 2]) * inv, __uint_as_float(ov[q4 * 8 + 3]) * inv);
          val.z = pack_bf16x2(__uint_as_float(ov[q4 * 8 + 4]) * inv, __uint_as_float(ov[q4 * 8 + 5]) * inv);
          val.w = pack_bf16x2(__uint_as_float(ov[q4 * 8 + 6]) * inv, __uint_as_float(ov[q4 * 8 + 7]) * inv);
          *reinterpret_cast<uint4*>(orow + c * 32 + q4 * 8) = val;
        }
      }
    }
    tc_fence_before();
  }

  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------ host
int make_tmap_2d_bf16(CUtensorMap* out, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_cols,
                      uint32_t box_rows);
int make_tmap_2d_f32(CUtensorMap* out, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_cols,
                     uint32_t box_rows);

template <int D>
static int attn_fwd_tc_launch(const void* q, const void* k, const void* v, void* o, float* lse, const int* cu, int nseq, int max_len,
                              int64_t ldq, int64_t ldk, int64_t ldv, int64_t ldo, int Hq, int Hkv, int T, float scale, cudaStream_t st) {
  using L = AttnFwdSmem<D>;
  auto kern = attn_fwd_tc_kernel<D>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::DYN);
    if (e != cudaSuccess) return set_error(B200_ERR_CUDA, "attn_fwd_tc smem attr: %s", cudaGetErrorString(e));
    configured = true;
  }
  CUtensorMap tq, tk, tv;
  int rc;
  if ((rc = make_tmap_2d_bf16(&tq, q, T, static_cast<uint64_t>(Hq) * D, ldq, 64, 128))) return rc;
  if ((rc = make_tmap_2d_bf16(&tk, k, T, static_cast<uint64_t>(Hkv) * D, ldk, 64, 128))) return rc;
  if ((rc = make_tmap_2d_bf16(&tv, v, T, static_cast<uint64_t>(Hkv) * D, ldv, 64, 128))) return rc;
  dim3 grid((max_len + 127) / 128, Hq, nseq);
  kern<<<grid, 320, L::DYN, st>>>(tq, tk, tv, static_cast<__nv_bfloat16*>(o), lse, cu, ldo, Hq, Hkv, T, scale * 1.4426950408889634f);
  B200_CHECK_LAUNCH("attn_fwd_tc");
  return 0;
}

int attn_fwd_tc(const void* q, const void* k, const void* v, void* o, float* lse, const int* cu_seqlens, int nseq, int max_len,
                int64_t ldq, int64_t ldk, int64_t ldv, int64_t ldo, int Hq, int Hkv, int D, int T, float scale, cudaStream_t st) {
  if (Hq % Hkv) return set_error(B200_ERR_ARG, "attn: Hq %% Hkv != 0");
  if ((ldq | ldk | ldv | ldo) % 8) return set_error(B200_ERR_ARG, "attn: row pitches must be multiples of 8 elements");
  if (D == 128) return attn_fwd_tc_launch<128>(q, k, v, o, lse, cu_seqlens, nseq, max_len, ldq, ldk, ldv, ldo, Hq, Hkv, T, scale, st);
  if (D == 64) return attn_fwd_tc_launch<64>(q, k, v, o, lse, cu_seqlens, nseq, max_len, ldq, ldk, ldv, ldo, Hq, Hkv, T, scale, st);
  return set_error(B200_ERR_UNSUPPORTED, "attn: head_dim %d not in {64,128}", D);
}

}  // namespace b200

// ================================================================================================ backward (tcgen05)
// CTA = one 128-row kv tile of one (sequence, kv head); loops over the q heads of the GQA group and the q tiles at or after
// the diagonal ("pairs").  Transposed orientation: S^T = K Q^T and dP^T = V dO^T put one KV ROW in each TMEM lane, so
//   P^T / dS^T written row-wise to 128B-swizzled smem are at once
//     - K-major A operands of  dV += P^T dO  and  dK += dS^T Q        (contraction over q), and
//     - the MN-major A operand of  dQ = dS K                          (same bytes, other descriptor: no transpose pass);
//   Q / dO / K tiles serve as K-major B (for S^T, dP^T) and as MN-major B (for dV, dK, dQ) from ONE copy in smem.
// TMEM (512 columns): S^T [0,128) | dP^T [128,256) (re-used by dQ after dP^T is consumed) | dV [256,256+D) | dK [384,384+D).
// dK / dV accumulate in TMEM over every pair of the CTA (GQA reduction included); dQ tiles are added to an fp32 buffer
// with 16-byte vector atomics.
namespace b200 {

#ifdef B200_ATTN_PROFILE
__device__ unsigned long long g_attn_prof[32];
#define PROF_DECL unsigned long long pt0 = clock64(), pt1
#define PROF(slot) do { pt1 = clock64(); if (blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) atomicAdd(&g_attn_prof[slot], pt1 - pt0); pt0 = pt1; } while (0)
#else
#define PROF_DECL
#define PROF(slot)
#endif

template <int D>
struct AttnBwdSmem {
  static constexpr int TILE = 128 * D * 2;
  static constexpr int PT_BYTES = 128 * 128 * 2;
  static constexpr int K_OFF = 0;
  static constexpr int V_OFF = TILE;
  static constexpr int Q_OFF = 2 * TILE;       // 2 stages
  static constexpr int DO_OFF = 4 * TILE;
  static constexpr int PT_OFF = 5 * TILE;
  static constexpr int DST_OFF = PT_OFF + PT_BYTES;
  static constexpr int LSE_OFF = DST_OFF + PT_BYTES;          // float [2][128] lse*log2e, then [2][128] delta
  static constexpr int BAR_OFF = LSE_OFF + 4 * 128 * 4;
  static constexpr int NUM_BARS = 1 + 2 + 2 + 1 + 1 + 1 + 1 + 1 + 1 + 1 + 4 + 1;  // kv_full, q_full[2], q_empty[2], do_full, do_empty, sdp_full, pt_ready, dq_full, dq_free, pa_ready, stage_free[4]
  static constexpr int DYN = BAR_OFF + NUM_BARS * 8 + 16;   // 231,528 B at D=128: no room for manual alignment slack
};

template <int D>
__global__ void __launch_bounds__(576, 1)  // 18 warps: 5 on two of the four schedulers -> at most 16384/(5*32) = 102 registers per thread
attn_bwd_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                   const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmDO,
                   const __grid_constant__ CUtensorMap tmDQ, const float* __restrict__ lse, const float* __restrict__ delta,
                   __nv_bfloat16* __restrict__ dk, __nv_bfloat16* __restrict__ dv, const int* __restrict__ cu_seqlens,
                   int64_t lddk, int64_t lddv, int Hq, int Hkv, int T, float scale, float scale_log2, int dq_cta_rows) {
  using L = AttnBwdSmem<D>;
  constexpr int ATOMS = D / 64;
  extern __shared__ __align__(1024) uint8_t smem[];
  if (smem_u32(smem) & 1023) __trap();  // 128B-swizzle atoms need a 1024-byte aligned base
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);
  uint64_t* kv_full = bars;
  uint64_t* q_full = bars + 1;
  uint64_t* q_empty = bars + 3;
  uint64_t* do_full = bars + 5;
  uint64_t* do_empty = bars + 6;
  uint64_t* sdp_full = bars + 7;
  uint64_t* pt_ready = bars + 8;
  uint64_t* dq_full = bars + 9;
  uint64_t* dq_free = bars + 10;
  uint64_t* pa_ready = bars + 11;
  uint64_t* kv_free = bars + 16;     // every MMA of a pass (readers of the K / V tiles) has completed
  uint64_t* stage_free = bars + 12;  // [4]: per lane quarter, the dQ staging (aliasing P^T / dS^T rows of that quarter) has been read by TMA
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bars + L::NUM_BARS);
  float* s_lse = reinterpret_cast<float*>(smem + L::LSE_OFF);  // [2][128]
  float* s_delta = s_lse + 256;                                 // [2][128]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int seq = blockIdx.z, hk = blockIdx.y;
  const int s0 = cu_seqlens[seq];
  const int len = cu_seqlens[seq + 1] - s0;
  const int G = Hq / Hkv;
  const int mt_end = (len + 127) / 128;  // kv / q tiles of this sequence
  // Causal load balance: CTA x takes kv tile x (mt_end - x q tiles per head) AND kv tile mt_end-1-x (x+1 q tiles): every CTA of a
  // sequence does the same number of (q tile, kv tile) pairs.
  if (static_cast<int>(blockIdx.x) >= (mt_end + 1) / 2) return;
  const int nt_pass[2] = {static_cast<int>(blockIdx.x), mt_end - 1 - static_cast<int>(blockIdx.x)};
  const int n_pass = nt_pass[0] == nt_pass[1] ? 1 : 2;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    tma_prefetch_desc(&tmDO);
    tma_prefetch_desc(&tmDQ);
    mbar_init(kv_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&q_full[i], 1);
      mbar_init(&q_empty[i], 1);
    }
    mbar_init(do_full, 1);
    mbar_init(do_empty, 1);
    mbar_init(sdp_full, 1);
    mbar_init(pt_ready, 16);
    mbar_init(pa_ready, 16);
    mbar_init(kv_free, 1);
    for (int i = 0; i < 4; ++i) mbar_init(&stage_free[i], D / 32);  // the OUT_CHUNKS warps of a lane quarter
    mbar_init(dq_full, 1);
    mbar_init(dq_free, D / 8);   // (D/32 column chunks) x 4 lane quarters
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_holder, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;
  const uint32_t tST = tmem_base, tDP = tmem_base + 128, tDV = tmem_base + 256, tDK = tmem_base + 384;

  if (warp == 0) {
    // ===================================================== TMA producer
    if (lane == 0) {
      int gp = 0;  // pairs issued so far over both passes (barrier parities / Q stages run on this global counter)
      for (int pass = 0; pass < n_pass; ++pass) {
        const int nt = nt_pass[pass], n0 = nt * 128;
        const int pairs_per_head = mt_end - nt, n_pairs = G * pairs_per_head;
        // every MMA of the previous pass (readers of K / V) has completed.  A dedicated once-per-pass barrier: this thread can be
        // two pairs ahead of the MMAs, so the per-pair dq_full parity would alias.
        if (pass > 0) mbar_wait(kv_free, (pass - 1) & 1);
        mbar_arrive_expect_tx(kv_full, 2 * L::TILE);
#pragma unroll
        for (int a = 0; a < ATOMS; ++a) {
          tma_load_2d(smem + L::K_OFF + a * 16384, &tmK, kv_full, hk * D + a * 64, s0 + n0);
          tma_load_2d(smem + L::V_OFF + a * 16384, &tmV, kv_full, hk * D + a * 64, s0 + n0);
        }
        int h = hk * G, mt = nt;
        for (int p = 0; p < n_pairs; ++p, ++gp) {
          const int m0 = mt * 128;
          const int st = gp & 1;
          mbar_wait(&q_empty[st], ((gp >> 1) & 1) ^ 1);
          mbar_arrive_expect_tx(&q_full[st], L::TILE);
#pragma unroll
          for (int a = 0; a < ATOMS; ++a) tma_load_2d(smem + L::Q_OFF + st * L::TILE + a * 16384, &tmQ, &q_full[st], h * D + a * 64, s0 + m0);
          mbar_wait(do_empty, (gp & 1) ^ 1);
          mbar_arrive_expect_tx(do_full, L::TILE);
#pragma unroll
          for (int a = 0; a < ATOMS; ++a) tma_load_2d(smem + L::DO_OFF + a * 16384, &tmDO, do_full, h * D + a * 64, s0 + m0);
          if (++mt == mt_end) {
            mt = nt;
            ++h;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================================================== MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc_st = make_idesc_bf16(128, 128, 0, 0);  // S^T = K Q^T, dP^T = V dO^T  (both operands K-major over d)
      constexpr uint32_t idesc_dkv = make_idesc_bf16(128, D, 0, 1);   // dV += P^T dO, dK += dS^T Q  (A K-major over q, B MN-major)
      constexpr uint32_t idesc_dq = make_idesc_bf16(128, D, 1, 1);    // dQ = dS K                   (A MN-major from dS^T, B MN-major)
      const uint32_t k_base = smem_u32(smem + L::K_OFF), v_base = smem_u32(smem + L::V_OFF);
      const uint32_t do_base = smem_u32(smem + L::DO_OFF);
      const uint32_t pt_base = smem_u32(smem + L::PT_OFF), dst_base = smem_u32(smem + L::DST_OFF);
      PROF_DECL;
      int gp = 0;
      for (int pass = 0; pass < n_pass; ++pass) {
        const int n_pairs = G * (mt_end - nt_pass[pass]);
        mbar_wait(kv_full, pass & 1);
        for (int p = 0; p < n_pairs; ++p, ++gp) {
          const int st = gp & 1;
          const uint32_t q_base = smem_u32(smem + L::Q_OFF + st * L::TILE);
          // S^T (the compute warps finished loading S^T of the previous pair before its pt_ready, which this thread has waited on)
          mbar_wait(&q_full[st], (gp >> 1) & 1);
          PROF(0);
          tc_fence_after();
#pragma unroll
          for (int kk = 0; kk < D / 16; ++kk) {
            const uint32_t off = (kk >> 2) * 16384 + (kk & 3) * 32;
            umma_bf16(tST, make_smem_desc_sw128(k_base + off, 16, 1024), make_smem_desc_sw128(q_base + off, 16, 1024), idesc_st, kk != 0);
          }
          // dP^T goes where the previous pair's dQ lives: wait until it has been read out
          PROF(1);
          mbar_wait(do_full, gp & 1);
          PROF(2);
          mbar_wait(dq_free, (gp & 1) ^ 1);
          PROF(3);
          tc_fence_after();
#pragma unroll
          for (int kk = 0; kk < D / 16; ++kk) {
            const uint32_t off = (kk >> 2) * 16384 + (kk & 3) * 32;
            umma_bf16(tDP, make_smem_desc_sw128(v_base + off, 16, 1024), make_smem_desc_sw128(do_base + off, 16, 1024), idesc_st, kk != 0);
          }
          umma_commit(sdp_full);
          PROF(4);
          mbar_wait(pa_ready, gp & 1);  // P^T is in smem (dS^T still being computed: dV overlaps it)
          tc_fence_after();
          // dV += P^T dO      A: P^T [kv x q] K-major (2 atoms of 64 q);  B: dO [q x d] MN-major.  p == 0 starts a fresh kv tile.
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_bf16(tDV, make_smem_desc_sw128(pt_base + (kk >> 2) * 16384 + (kk & 3) * 32, 16, 1024),
                      make_smem_desc_sw128(do_base + kk * 2048, 16384, 1024), idesc_dkv, (p | kk) != 0);
          umma_commit(do_empty);
          mbar_wait(pt_ready, gp & 1);
          PROF(5);
          tc_fence_after();
          // dK += dS^T Q
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_bf16(tDK, make_smem_desc_sw128(dst_base + (kk >> 2) * 16384 + (kk & 3) * 32, 16, 1024),
                      make_smem_desc_sw128(q_base + kk * 2048, 16384, 1024), idesc_dkv, (p | kk) != 0);
          umma_commit(&q_empty[st]);
          // dQ = dS K         A: dS from the dS^T tile read MN-major (M = q contiguous, K = kv rows);  B: K [kv x d] MN-major
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_bf16(tDP, make_smem_desc_sw128(dst_base + kk * 2048, 16384, 1024), make_smem_desc_sw128(k_base + kk * 2048, 16384, 1024),
                      idesc_dq, kk != 0);
          umma_commit(dq_full);
          PROF(6);
        }
        umma_commit(kv_free);
      }
    }
  } else {
    // ===================================================== 16 compute warps.  Warp (quad, chunk): TMEM lanes [32*quad, +32) x 32 columns
    // [32*chunk, +32).  Thread <-> kv row n0+r (S^T, dP^T, dK, dV) and q row m0+r (dQ).  Four warps per scheduler hide the
    // TMEM / MUFU / shared-memory latencies that a single warp per scheduler exposes.
    const int cw = warp - 2;         // 0..15
    const int quad = warp & 3;       // TMEM lane quarter this warp may access (warp id % 4)
    const int chunk = cw >> 2;       // 0..3
    const int r = quad * 32 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(quad * 32) << 16;
    const int ct = threadIdx.x - 64;  // 0..511; the first 128 stage the per-q statistics
    constexpr float LOG2E = 1.4426950408889634f;
    constexpr int OUT_CHUNKS = D / 32;  // column chunks of the dQ / dK / dV tiles
    uint8_t* pt_row = smem + L::PT_OFF + r * 128;
    uint8_t* dst_row = smem + L::DST_OFF + r * 128;
#ifdef B200_ATTN_PROFILE
    unsigned long long pt0 = clock64(), pt1;
#define CPROF(slot) do { if (warp == 2 && lane == 0) { pt1 = clock64(); if (blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) atomicAdd(&g_attn_prof[slot], pt1 - pt0); pt0 = pt1; } } while (0)
#else
#define CPROF(slot)
#endif
    int gp = 0;  // global pair counter over both passes (barrier parities)
    for (int pass = 0; pass < n_pass; ++pass) {
    const int nt = nt_pass[pass], n0 = nt * 128;
    const int n_pairs = G * (mt_end - nt);
    const int kv = n0 + r;
    // per-q statistics (lse*log2e, delta) of the NEXT pair are fetched one pair ahead into registers of the first 128 threads
    float nxt_lse = 0.f, nxt_dlt = 0.f;
    if (ct < 128) {
      const int qi = nt * 128 + ct;  // pair 0: head hk*G, q tile nt
      if (qi < len) {
        nxt_lse = lse[static_cast<int64_t>(hk * G) * T + s0 + qi] * LOG2E;
        nxt_dlt = delta[static_cast<int64_t>(hk * G) * T + s0 + qi];
      }
    }
    int h = hk * G, mt = nt;
    for (int p = 0; p < n_pairs; ++p, ++gp) {
      const int m0 = mt * 128;
      int h_n = h, mt_n = mt + 1;
      if (mt_n == mt_end) {
        mt_n = nt;
        ++h_n;
      }
      float* lse2 = s_lse + (gp & 1) * 128;
      float* dlt = s_delta + (gp & 1) * 128;
      if (ct < 128) {
        lse2[ct] = nxt_lse;
        dlt[ct] = nxt_dlt;
        nxt_lse = nxt_dlt = 0.f;
        const int qi = mt_n * 128 + ct;
        if (p + 1 < n_pairs && qi < len) {
          nxt_lse = lse[static_cast<int64_t>(h_n) * T + s0 + qi] * LOG2E;
          nxt_dlt = delta[static_cast<int64_t>(h_n) * T + s0 + qi];
        }
      }
      asm volatile("bar.sync 1, 512;" ::: "memory");
      CPROF(8);
      const bool need_mask = (mt == nt) || (m0 + 128 > len) || (n0 + 128 > len);
      mbar_wait(sdp_full, gp & 1);
      CPROF(9);
      tc_fence_after();
      {
        const int c = chunk;  // this warp's 32 q columns
        uint32_t sv[32];
        tmem_ld_32x32b_x32(tST + lane_addr + c * 32, sv);
        tmem_ld_wait();
        // ---- phase A: P^T = 2^(S^T * scale*log2e - lse*log2e)  -> smem; the MMA warp starts dV += P^T dO right away
        const float4* l4 = reinterpret_cast<const float4*>(lse2 + c * 32);
        float pf[32];
#pragma unroll
        for (int e4 = 0; e4 < 8; ++e4) {
          const float4 ls = l4[e4];
          pf[e4 * 4 + 0] = ex2_approx(__uint_as_float(sv[e4 * 4 + 0]) * scale_log2 - ls.x);
          pf[e4 * 4 + 1] = ex2_approx(__uint_as_float(sv[e4 * 4 + 1]) * scale_log2 - ls.y);
          pf[e4 * 4 + 2] = ex2_approx(__uint_as_float(sv[e4 * 4 + 2]) * scale_log2 - ls.z);
          pf[e4 * 4 + 3] = ex2_approx(__uint_as_float(sv[e4 * 4 + 3]) * scale_log2 - ls.w);
        }
        if (need_mask) {
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const int qc = m0 + c * 32 + e;
            if (qc < kv || qc >= len || kv >= len) pf[e] = 0.f;
          }
        }
        // the previous pair's dQ staging lives in these P^T / dS^T rows: its TMA reduce must have finished READING them.
        // Checked only now, after the exp work, so the reduction drains behind it instead of on the critical path.
        if (chunk < OUT_CHUNKS) {
          if (lane == 0) {
            tma_store_wait_read<0>();
            mbar_arrive(&stage_free[quad]);
          }
        }
        mbar_wait(&stage_free[quad], gp & 1);
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {
          const int ch = c * 4 + q4;  // 16-byte chunk = 8 q columns; atom = ch / 8
          const uint32_t off = (ch >> 3) * 16384 + (((ch & 7) ^ (r & 7)) << 4);
          *reinterpret_cast<uint4*>(pt_row + off) =
              make_uint4(pack_bf16x2(pf[q4 * 8 + 0], pf[q4 * 8 + 1]), pack_bf16x2(pf[q4 * 8 + 2], pf[q4 * 8 + 3]),
                         pack_bf16x2(pf[q4 * 8 + 4], pf[q4 * 8 + 5]), pack_bf16x2(pf[q4 * 8 + 6], pf[q4 * 8 + 7]));
        }
        tc_fence_before();
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(pa_ready);
        // ---- phase B: dS^T = P^T * (dP^T - delta) -> smem
        uint32_t dv_[32];
        tmem_ld_32x32b_x32(tDP + lane_addr + c * 32, dv_);
        tmem_ld_wait();
        const float4* d4 = reinterpret_cast<const float4*>(dlt + c * 32);
#pragma unroll
        for (int e4 = 0; e4 < 8; ++e4) {
          const float4 dl = d4[e4];
          pf[e4 * 4 + 0] *= __uint_as_float(dv_[e4 * 4 + 0]) - dl.x;
          pf[e4 * 4 + 1] *= __uint_as_float(dv_[e4 * 4 + 1]) - dl.y;
          pf[e4 * 4 + 2] *= __uint_as_float(dv_[e4 * 4 + 2]) - dl.z;
          pf[e4 * 4 + 3] *= __uint_as_float(dv_[e4 * 4 + 3]) - dl.w;
        }
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {
          const int ch = c * 4 + q4;
          const uint32_t off = (ch >> 3) * 16384 + (((ch & 7) ^ (r & 7)) << 4);
          *reinterpret_cast<uint4*>(dst_row + off) =
              make_uint4(pack_bf16x2(pf[q4 * 8 + 0], pf[q4 * 8 + 1]), pack_bf16x2(pf[q4 * 8 + 2], pf[q4 * 8 + 3]),
                         pack_bf16x2(pf[q4 * 8 + 4], pf[q4 * 8 + 5]), pack_bf16x2(pf[q4 * 8 + 6], pf[q4 * 8 + 7]));
        }
      }
      tc_fence_before();
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(pt_ready);
      CPROF(10);
      // dQ tile of this pair (lane r = q row m0 + r).  Every warp waits (the next pair overwrites P^T / dS^T); the OUT_CHUNKS*4
      // warps that own a column chunk copy it TMEM -> registers -> swizzled fp32 staging (the now idle P^T/dS^T buffers) and
      // ONE thread per chunk issues a TMA reduce-add of the [128 x 32] fp32 box into the dq accumulator: 4 bulk L2 reductions per
      // pair instead of 4096 vector atomics.  Rows past the sequence end carry exact zeros (their dS is masked).
      mbar_wait(dq_full, gp & 1);
      CPROF(11);
      if (chunk < OUT_CHUNKS) {
        tc_fence_after();
        uint32_t qv[32];
        tmem_ld_32x32b_x32(tDP + lane_addr + chunk * 32, qv);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(dq_free);  // the dP^T / dQ columns may be overwritten by dP^T_{p+1}
        uint8_t* stage = smem + L::PT_OFF + chunk * 16384 + r * 128;
#pragma unroll
        for (int q4 = 0; q4 < 8; ++q4)
          *reinterpret_cast<uint4*>(stage + ((q4 ^ (r & 7)) << 4)) = make_uint4(qv[q4 * 4], qv[q4 * 4 + 1], qv[q4 * 4 + 2], qv[q4 * 4 + 3]);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {  // one [32 rows x 32 floats] box per warp: no cross-warp barrier, 16 reductions in flight per CTA
          tma_reduce_add_2d(&tmDQ, smem + L::PT_OFF + chunk * 16384 + quad * 4096, h * D + chunk * 32,
                            static_cast<int>(blockIdx.x) * dq_cta_rows + s0 + m0 + quad * 32);
          tma_store_commit();
        }
      }
      CPROF(12);
      h = h_n;
      mt = mt_n;
    }
    if (chunk < OUT_CHUNKS && lane == 0) tma_store_wait<0>();
    // dK (scaled) / dV rows of this kv tile; dq_full of the pass's last pair covers every MMA of the pass.  The next pass's first
    // dV / dK MMAs (accumulate = 0) are issued only after these warps have moved on to its first pair (pa_ready), i.e. after this read.
    mbar_wait(dq_full, (gp - 1) & 1);
    if (chunk < OUT_CHUNKS) {
      tc_fence_after();
      const bool valid = kv < len;  // tcgen05.ld is warp-collective: every lane loads, only valid rows store
      __nv_bfloat16* dkr = dk + static_cast<int64_t>(s0 + kv) * lddk + hk * D + chunk * 32;
      __nv_bfloat16* dvr = dv + static_cast<int64_t>(s0 + kv) * lddv + hk * D + chunk * 32;
      uint32_t a[32], b[32];
      tmem_ld_32x32b_x32(tDK + lane_addr + chunk * 32, a);
      tmem_ld_32x32b_x32(tDV + lane_addr + chunk * 32, b);
      tmem_ld_wait();
      if (valid) {
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {
          uint4 x, y;
          x.x = pack_bf16x2(__uint_as_float(a[q4 * 8 + 0]) * scale, __uint_as_float(a[q4 * 8 + 1]) * scale);
          x.y = pack_bf16x2(__uint_as_float(a[q4 * 8 + 2]) * scale, __uint_as_float(a[q4 * 8 + 3]) * scale);
          x.z = pack_bf16x2(__uint_as_float(a[q4 * 8 + 4]) * scale, __uint_as_float(a[q4 * 8 + 5]) * scale);
          x.w = pack_bf16x2(__uint_as_float(a[q4 * 8 + 6]) * scale, __uint_as_float(a[q4 * 8 + 7]) * scale);
          y.x = pack_bf16x2(__uint_as_float(b[q4 * 8 + 0]), __uint_as_float(b[q4 * 8 + 1]));
          y.y = pack_bf16x2(__uint_as_float(b[q4 * 8 + 2]), __uint_as_float(b[q4 * 8 + 3]));
          y.z = pack_bf16x2(__uint_as_float(b[q4 * 8 + 4]), __uint_as_float(b[q4 * 8 + 5]));
          y.w = pack_bf16x2(__uint_as_float(b[q4 * 8 + 6]), __uint_as_float(b[q4 * 8 + 7]));
          *reinterpret_cast<uint4*>(dkr + q4 * 8) = x;
          *reinterpret_cast<uint4*>(dvr + q4 * 8) = y;
        }
      }
      tc_fence_before();
    }
    }  // pass
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

int attn_delta_launch(const void* o, const void* dout, float* delta, int64_t ldo, int64_t lddo, int Hq, int D, int T, cudaStream_t st);
int attn_dq_convert_launch(const float* acc, int nbuf, void* dq, int64_t T, int cols, int64_t lddq, float scale, cudaStream_t st);

template <int D>
static int attn_bwd_tc_launch(const void* q, const void* k, const void* v, const void* o, const void* dout, const float* lse, void* dq,
                              void* dk, void* dv, void* ws, size_t ws_bytes, const int* cu, int nseq, int max_len, int64_t ldq, int64_t ldk,
                              int64_t ldv, int64_t ldo, int64_t lddo, int64_t lddq, int64_t lddk, int64_t lddv, int Hq, int Hkv, int T,
                              float scale, cudaStream_t st) {
  using L = AttnBwdSmem<D>;
  auto kern = attn_bwd_tc_kernel<D>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::DYN);
    if (e != cudaSuccess) return set_error(B200_ERR_CUDA, "attn_bwd_tc smem attr: %s", cudaGetErrorString(e));
    configured = true;
  }
  // The dQ tiles of one (sequence, kv head) come from `pairs` CTAs, and each CTA adds at most two tiles to an element (one per kv tile
  // it owns), so with one fp32 accumulator per CTA every element is summed in a fixed order and dQ is bit-reproducible.  That costs
  // `pairs` accumulators of memset and read-back, so it is done for two CTAs (longest sequence 257..512 tokens) when the caller sized
  // the workspace for it (attn_bwd_workspace_bytes with max_seqlen <= 512); otherwise the CTAs share one accumulator and the order of
  // the fp32 additions follows their timing (last-bit differences from launch to launch).  One CTA adds at most two tiles anyway.
  const int pairs = ((max_len + 127) / 128 + 1) / 2;
  const size_t acc_elems = static_cast<size_t>(T) * Hq * D;
  const size_t delta_bytes = static_cast<size_t>(T) * Hq * sizeof(float);
  if (ws_bytes < acc_elems * sizeof(float) + delta_bytes) return set_error(B200_ERR_ARG, "attn_bwd: workspace of %zu bytes is too small", ws_bytes);
  const int nbuf = pairs == 2 && ws_bytes >= 2 * acc_elems * sizeof(float) + delta_bytes ? 2 : 1;
  float* dq_acc = static_cast<float*>(ws);
  float* delta = dq_acc + nbuf * acc_elems;
  cudaError_t e = cudaMemsetAsync(dq_acc, 0, nbuf * acc_elems * sizeof(float), st);
  if (e != cudaSuccess) return set_error(B200_ERR_CUDA, "attn_bwd memset: %s", cudaGetErrorString(e));
  int rc;
  if ((rc = attn_delta_launch(o, dout, delta, ldo, lddo, Hq, D, T, st))) return rc;
  CUtensorMap tq, tk, tv, tdo, tdq;
  if ((rc = make_tmap_2d_f32(&tdq, dq_acc, static_cast<uint64_t>(nbuf) * T, static_cast<uint64_t>(Hq) * D, static_cast<uint64_t>(Hq) * D, 32, 32))) return rc;
  if ((rc = make_tmap_2d_bf16(&tq, q, T, static_cast<uint64_t>(Hq) * D, ldq, 64, 128))) return rc;
  if ((rc = make_tmap_2d_bf16(&tk, k, T, static_cast<uint64_t>(Hkv) * D, ldk, 64, 128))) return rc;
  if ((rc = make_tmap_2d_bf16(&tv, v, T, static_cast<uint64_t>(Hkv) * D, ldv, 64, 128))) return rc;
  if ((rc = make_tmap_2d_bf16(&tdo, dout, T, static_cast<uint64_t>(Hq) * D, lddo, 64, 128))) return rc;
  dim3 grid(((max_len + 127) / 128 + 1) / 2, Hkv, nseq);
  kern<<<grid, 576, L::DYN, st>>>(tq, tk, tv, tdo, tdq, lse, delta, static_cast<__nv_bfloat16*>(dk), static_cast<__nv_bfloat16*>(dv), cu,
                                  lddk, lddv, Hq, Hkv, T, scale, scale * 1.4426950408889634f, nbuf > 1 ? T : 0);
  B200_CHECK_LAUNCH("attn_bwd_tc");
#ifdef B200_ATTN_PROFILE
  {
    cudaStreamSynchronize(st);
    unsigned long long h[32];
    cudaMemcpyFromSymbol(h, g_attn_prof, sizeof(h));
    static const char* names[] = {"mma:wait q_full", "mma:issue S^T", "mma:wait do_full", "mma:wait dq_free", "mma:issue dP^T", "mma:wait pt_ready",
                                  "mma:issue dV,dK,dQ", "", "cmp:stats+bar", "cmp:wait sdp_full", "cmp:compute+store", "cmp:wait dq_full", "cmp:dq readout"};
    const int npairs = (Hq / Hkv) * ((max_len + 127) / 128 + 1);
    for (int i = 0; i < 13; ++i) if (names[i][0]) fprintf(stderr, "ATTN_PROF %-22s %8.0f cycles/pair\n", names[i], double(h[i]) / npairs);
    unsigned long long z[32] = {0};
    cudaMemcpyToSymbol(g_attn_prof, z, sizeof(z));
  }
#endif
  return attn_dq_convert_launch(dq_acc, nbuf, dq, T, Hq * D, lddq, scale, st);
}

int attn_bwd_tc(const void* q, const void* k, const void* v, const void* o, const void* dout, const float* lse, void* dq, void* dk,
                void* dv, void* ws, size_t ws_bytes, const int* cu_seqlens, int nseq, int max_len, int64_t ldq, int64_t ldk, int64_t ldv,
                int64_t ldo, int64_t lddo, int64_t lddq, int64_t lddk, int64_t lddv, int Hq, int Hkv, int D, int T, float scale, cudaStream_t st) {
  if (Hq % Hkv) return set_error(B200_ERR_ARG, "attn: Hq %% Hkv != 0");
  if ((ldq | ldk | ldv | ldo | lddo | lddq | lddk | lddv) % 8) return set_error(B200_ERR_ARG, "attn: row pitches must be multiples of 8 elements");
  if (D == 128)
    return attn_bwd_tc_launch<128>(q, k, v, o, dout, lse, dq, dk, dv, ws, ws_bytes, cu_seqlens, nseq, max_len, ldq, ldk, ldv, ldo, lddo, lddq, lddk,
                                   lddv, Hq, Hkv, T, scale, st);
  if (D == 64)
    return attn_bwd_tc_launch<64>(q, k, v, o, dout, lse, dq, dk, dv, ws, ws_bytes, cu_seqlens, nseq, max_len, ldq, ldk, ldv, ldo, lddo, lddq, lddk,
                                  lddv, Hq, Hkv, T, scale, st);
  return set_error(B200_ERR_UNSUPPORTED, "attn: head_dim %d not in {64,128}", D);
}

}  // namespace b200
