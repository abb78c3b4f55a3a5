// Causal GQA flash attention, forward + backward, variable-length (packed) sequences via cu_seqlens.
// Token-major layout: q [T, Hq*D] (row pitch ldq), k/v [T, Hkv*D], o [T, Hq*D]; lse [Hq, T] fp32 (natural log).
// Restates what the reference reaches through ALL_ATTENTION_FUNCTIONS[...] (flash-attn / SDPA):
//   /root/reference/nemo_automodel/components/models/llama/model.py:135-148 (causal, GQA, scale = D^-0.5, dropout 0);
//   packed sequences = block-diagonal causal mask (components/datasets/llm/packed_sequence.py position_ids restart).
// Online-softmax tiling (one 64-row q tile per CTA, 64-row kv tiles), fp32 accumulate, P rounded to bf16 for P*V.
// v1 uses warp-level mma.sync.m16n8k16 tensor-core instructions; the tcgen05/TMEM version is the planned upgrade.
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <math.h>

#include "common.h"
#include "ptx.cuh"

namespace b200 {

// ------------------------------------------------------------------------------------------------ primitives
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, bool pred) {
  const int sz = pred ? 16 : 0;  // src-size 0 => zero fill
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// smem tile [rows][D] bf16, 16B chunks XOR-swizzled by (row & 7): conflict-free ldmatrix and cp.async
template <int D>
__device__ __forceinline__ uint32_t tile_off(int row, int chunk) {
  return static_cast<uint32_t>(row * (D * 2) + ((chunk ^ (row & 7)) << 4));
}

// load a [64][D] tile (rows row0.. of a token-major tensor) into swizzled smem; rows >= nrows_valid are zero-filled
template <int D, int THREADS>
__device__ __forceinline__ void load_tile(uint32_t smem_base, const __nv_bfloat16* gbase, int64_t ld, int row0, int nrows_valid) {
  constexpr int CH = D / 8;
#pragma unroll
  for (int i = threadIdx.x; i < 64 * CH; i += THREADS) {
    const int r = i / CH, c = i % CH;
    const bool ok = (row0 + r) < nrows_valid;
    const __nv_bfloat16* src = gbase + static_cast<int64_t>(ok ? (row0 + r) : 0) * ld + c * 8;
    cp_async16(smem_base + tile_off<D>(r, c), src, ok);
  }
}

// A fragment (16 rows x 16 k) from a row-major [m][k] tile
template <int D>
__device__ __forceinline__ void ld_A(uint32_t (&a)[4], uint32_t base, int row0, int k0, int lane) {
  ldsm_x4(a, base + tile_off<D>(row0 + (lane & 15), (k0 >> 3) + (lane >> 4)));
}
// B fragments for two adjacent n-tiles (16 n) x 16 k from [n][k] storage (non-transposed): {b0,b1 of nt0, b0,b1 of nt1}
template <int D>
__device__ __forceinline__ void ld_B_nk(uint32_t (&b)[4], uint32_t base, int n0, int k0, int lane) {
  ldsm_x4(b, base + tile_off<D>(n0 + (lane & 7) + ((lane >> 4) << 3), (k0 >> 3) + ((lane >> 3) & 1)));
}
// B fragments for two adjacent n-tiles x 16 k from [k][n] storage (transposed load)
template <int D>
__device__ __forceinline__ void ld_B_kn(uint32_t (&b)[4], uint32_t base, int k0, int n0, int lane) {
  ldsm_x4_t(b, base + tile_off<D>(k0 + (lane & 7) + (((lane >> 3) & 1) << 3), (n0 >> 3) + (lane >> 4)));
}
// A fragment (16 m x 16 k) from [k][m] storage (transposed load)
template <int D>
__device__ __forceinline__ void ld_A_km(uint32_t (&a)[4], uint32_t base, int m0, int k0, int lane) {
  ldsm_x4_t(a, base + tile_off<D>(k0 + (lane & 7) + ((lane >> 4) << 3), (m0 >> 3) + ((lane >> 3) & 1)));
}

// ------------------------------------------------------------------------------------------------ forward
template <int D>
__global__ void __launch_bounds__(128) attn_fwd_kernel(const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ k,
                                                      const __nv_bfloat16* __restrict__ v, __nv_bfloat16* __restrict__ o,
                                                      float* __restrict__ lse, const int* __restrict__ cu_seqlens, int64_t ldq,
                                                      int64_t ldk, int64_t ldv, int64_t ldo, int Hq, int Hkv, int T,
                                                      float scale_log2) {
  constexpr int BM = 64, BN = 64, TILE = 64 * D * 2;
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sQ = smem_u32(smem), sK = sQ + TILE, sV = sK + TILE;
  const int seq = blockIdx.z, h = blockIdx.y;
  const int mt = gridDim.x - 1 - blockIdx.x;  // heavy (late) tiles first
  const int s0 = cu_seqlens[seq];
  const int len = cu_seqlens[seq + 1] - s0;
  const int m0 = mt * BM;
  if (m0 >= len) return;
  const int hk = h / (Hq / Hkv);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const __nv_bfloat16* qb = q + static_cast<int64_t>(s0) * ldq + h * D;
  const __nv_bfloat16* kb = k + static_cast<int64_t>(s0) * ldk + hk * D;
  const __nv_bfloat16* vb = v + static_cast<int64_t>(s0) * ldv + hk * D;

  load_tile<D, 128>(sQ, qb, ldq, m0, len);
  load_tile<D, 128>(sK, kb, ldk, 0, len);
  cp_async_commit();

  float o_acc[D / 8][4];
#pragma unroll
  for (int i = 0; i < D / 8; ++i)
#pragma unroll
    for (int e = 0; e < 4; ++e) o_acc[i][e] = 0.f;
  float row_m[2] = {-INFINITY, -INFINITY}, row_l[2] = {0.f, 0.f};
  uint32_t qf[D / 16][4];

  const int nj = mt + 1;  // causal: kv tiles 0..mt (BM == BN)
  const int r_lo = m0 + warp * 16 + (lane >> 2);  // this thread's two q rows (sequence-relative): r_lo, r_lo + 8
  for (int j = 0; j < nj; ++j) {
    cp_async_wait<0>();
    __syncthreads();  // K_j (and Q) landed; every warp is done with V_{j-1}
    load_tile<D, 128>(sV, vb, ldv, j * BN, len);
    cp_async_commit();
    if (j == 0) {
#pragma unroll
      for (int kk = 0; kk < D / 16; ++kk) ld_A<D>(qf[kk], sQ, warp * 16, kk * 16, lane);
    }
    float s[BN / 8][4];
#pragma unroll
    for (int i = 0; i < BN / 8; ++i)
#pragma unroll
      for (int e = 0; e < 4; ++e) s[i][e] = 0.f;
#pragma unroll
    for (int kk = 0; kk < D / 16; ++kk) {
#pragma unroll
      for (int np = 0; np < BN / 16; ++np) {
        uint32_t b[4];
        ld_B_nk<D>(b, sK, np * 16, kk * 16, lane);
        mma16816(s[2 * np], qf[kk], b[0], b[1]);
        mma16816(s[2 * np + 1], qf[kk], b[2], b[3]);
      }
    }
    // mask (diagonal tile and the sequence tail), scale into log2 domain
    const bool need_mask = (j == nj - 1) || ((j + 1) * BN > len);
#pragma unroll
    for (int i = 0; i < BN / 8; ++i) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int col = j * BN + i * 8 + ((lane & 3) << 1) + (e & 1);
        const int row = r_lo + ((e >> 1) << 3);
        float x = s[i][e] * scale_log2;
        if (need_mask && (col > row || col >= len)) x = -INFINITY;
        s[i][e] = x;
      }
    }
    // online softmax (rows live in a quad of 4 lanes)
#pragma unroll
    for (int hrow = 0; hrow < 2; ++hrow) {
      float mx = -INFINITY;
#pragma unroll
      for (int i = 0; i < BN / 8; ++i) mx = fmaxf(mx, fmaxf(s[i][2 * hrow], s[i][2 * hrow + 1]));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
      const float m_new = fmaxf(row_m[hrow], mx);
      const float m_use = (m_new == -INFINITY) ? 0.f : m_new;
      const float corr = exp2f(row_m[hrow] - m_use);  // row_m=-inf -> 0
      float sum = 0.f;
#pragma unroll
      for (int i = 0; i < BN / 8; ++i) {
        const float p0 = exp2f(s[i][2 * hrow] - m_use), p1 = exp2f(s[i][2 * hrow + 1] - m_use);
        s[i][2 * hrow] = p0;
        s[i][2 * hrow + 1] = p1;
        sum += p0 + p1;
      }
      row_l[hrow] = row_l[hrow] * corr + sum;  // per-thread partial sums; quad-reduced at the end
      row_m[hrow] = m_new;
#pragma unroll
      for (int i = 0; i < D / 8; ++i) {
        o_acc[i][2 * hrow] *= corr;
        o_acc[i][2 * hrow + 1] *= corr;
      }
    }
    cp_async_wait<0>();
    __syncthreads();  // V_j landed; every warp is done reading K_j
    if (j + 1 < nj) {
      load_tile<D, 128>(sK, kb, ldk, (j + 1) * BN, len);
      cp_async_commit();
    }
#pragma unroll
    for (int kk = 0; kk < BN / 16; ++kk) {
      uint32_t a[4];
      a[0] = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]);
      a[1] = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
      a[2] = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
      a[3] = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
      for (int np = 0; np < D / 16; ++np) {
        uint32_t b[4];
        ld_B_kn<D>(b, sV, kk * 16, np * 16, lane);
        mma16816(o_acc[2 * np], a, b[0], b[1]);
        mma16816(o_acc[2 * np + 1], a, b[2], b[3]);
      }
    }
  }
  // finalize: normalise, stage through this warp's rows of sQ, coalesced 16B stores
#pragma unroll
  for (int hrow = 0; hrow < 2; ++hrow) {
    float l = row_l[hrow];
    l += __shfl_xor_sync(0xffffffffu, l, 1);
    l += __shfl_xor_sync(0xffffffffu, l, 2);
    const float inv = l > 0.f ? 1.f / l : 0.f;
    const int row = r_lo + hrow * 8;
    if ((lane & 3) == 0 && row < len) lse[static_cast<int64_t>(h) * T + s0 + row] = (row_m[hrow] + log2f(l)) * 0.6931471805599453f;
#pragma unroll
    for (int i = 0; i < D / 8; ++i) {
      o_acc[i][2 * hrow] *= inv;
      o_acc[i][2 * hrow + 1] *= inv;
    }
  }
  __syncwarp();
#pragma unroll
  for (int i = 0; i < D / 8; ++i) {
#pragma unroll
    for (int hrow = 0; hrow < 2; ++hrow) {
      const int r = warp * 16 + (lane >> 2) + hrow * 8;
      const uint32_t addr = sQ + tile_off<D>(r, i) + ((lane & 3) << 2);
      const uint32_t val = pack_bf16x2(o_acc[i][2 * hrow], o_acc[i][2 * hrow + 1]);
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(val) : "memory");
    }
  }
  __syncwarp();
  constexpr int CH = D / 8;
  __nv_bfloat16* ob = o + static_cast<int64_t>(s0) * ldo + h * D;
  for (int i = lane; i < 16 * CH; i += 32) {
    const int r = warp * 16 + i / CH, c = i % CH;
    if (m0 + r < len) {
      uint4 val;
      asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(val.x), "=r"(val.y), "=r"(val.z), "=r"(val.w) : "r"(sQ + tile_off<D>(r, c)));
      *reinterpret_cast<uint4*>(ob + static_cast<int64_t>(m0 + r) * ldo + c * 8) = val;
    }
  }
}

// ------------------------------------------------------------------------------------------------ backward
// delta[h, t] = sum_d dO[t,h,d] * O[t,h,d].   D/8 lanes per (t, h) row, one 16-byte load of each operand per lane.
__global__ void __launch_bounds__(256) attn_delta_kernel(const __nv_bfloat16* __restrict__ o, const __nv_bfloat16* __restrict__ dout,
                                                        float* __restrict__ delta, int64_t ldo, int64_t lddo, int Hq, int D, int T) {
  const int lpr = D >> 3;                                   // lanes per row: 16 (D = 128) or 8 (D = 64)
  const int64_t gt = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  const int64_t r = gt / lpr;                               // row = t * Hq + h
  const int c = static_cast<int>(gt - r * lpr);
  float s = 0.f;
  const bool live = r < static_cast<int64_t>(T) * Hq;
  int t = 0, h = 0;
  if (live) {
    t = static_cast<int>(r / Hq);
    h = static_cast<int>(r - static_cast<int64_t>(t) * Hq);
    const uint4 a = *reinterpret_cast<const uint4*>(o + static_cast<int64_t>(t) * ldo + h * D + c * 8);
    const uint4 b = *reinterpret_cast<const uint4*>(dout + static_cast<int64_t>(t) * lddo + h * D + c * 8);
    const __nv_bfloat162* pa = reinterpret_cast<const __nv_bfloat162*>(&a);
    const __nv_bfloat162* pb = reinterpret_cast<const __nv_bfloat162*>(&b);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 x = __bfloat1622float2(pa[e]);
      const float2 y = __bfloat1622float2(pb[e]);
      s += x.x * y.x + x.y * y.y;
    }
  }
  for (int off = lpr >> 1; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);   // lpr is a power of two <= 32
  if (live && c == 0) delta[static_cast<int64_t>(h) * T + t] = s;
}

// One CTA per (kv tile of 64 rows, kv head, sequence).  Loops over the q heads of the GQA group and the q tiles at or
// after the diagonal.  Works in the transposed orientation (S^T = K Q^T: each warp owns 16 kv rows x 64 q columns) so P^T and
// dS^T are directly the A operands of dV += P^T dO and dK += dS^T Q; dS^T goes through smem once for dQ += dS K.
// dK/dV are reduced over the group's q heads in registers (no atomics); dQ is accumulated in fp32 with vector atomics.
template <int D>
__global__ void __launch_bounds__(128) attn_bwd_kernel(const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ k,
                                                      const __nv_bfloat16* __restrict__ v, const __nv_bfloat16* __restrict__ dout,
                                                      const float* __restrict__ lse, const float* __restrict__ delta,
                                                      float* __restrict__ dq_acc, __nv_bfloat16* __restrict__ dk,
                                                      __nv_bfloat16* __restrict__ dv, const int* __restrict__ cu_seqlens,
                                                      int64_t ldq, int64_t ldk, int64_t ldv, int64_t lddo, int64_t lddq,
                                                      int64_t lddk, int64_t lddv, int Hq, int Hkv, int T, float scale,
                                                      float scale_log2) {
  constexpr int BM = 64, BN = 64, TILE = 64 * D * 2;
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sK = smem_u32(smem), sV = sK + TILE, sQ = sV + TILE, sdO = sQ + TILE, sdS = sdO + TILE;
  float* s_lse = reinterpret_cast<float*>(smem + 4 * TILE + 64 * 64 * 2);
  float* s_delta = s_lse + 64;
  const int seq = blockIdx.z, hk = blockIdx.y, nt = blockIdx.x;
  const int s0 = cu_seqlens[seq];
  const int len = cu_seqlens[seq + 1] - s0;
  const int n0 = nt * BN;
  if (n0 >= len) return;
  const int G = Hq / Hkv;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const __nv_bfloat16* kb = k + static_cast<int64_t>(s0) * ldk + hk * D;
  const __nv_bfloat16* vb = v + static_cast<int64_t>(s0) * ldv + hk * D;
  load_tile<D, 128>(sK, kb, ldk, n0, len);
  load_tile<D, 128>(sV, vb, ldv, n0, len);
  cp_async_commit();

  float dk_acc[D / 8][4], dv_acc[D / 8][4];
#pragma unroll
  for (int i = 0; i < D / 8; ++i)
#pragma unroll
    for (int e = 0; e < 4; ++e) dk_acc[i][e] = dv_acc[i][e] = 0.f;

  const int mt_end = (len + BM - 1) / BM;
  const int kv_lo = n0 + warp * 16 + (lane >> 2);  // this thread's kv rows: kv_lo, kv_lo + 8
  constexpr float LOG2E = 1.4426950408889634f;

  for (int g = 0; g < G; ++g) {
    const int h = hk * G + g;
    const __nv_bfloat16* qb = q + static_cast<int64_t>(s0) * ldq + h * D;
    const __nv_bfloat16* dob = dout + static_cast<int64_t>(s0) * lddo + h * D;
    for (int mt = nt; mt < mt_end; ++mt) {
      const int m0 = mt * BM;
      __syncthreads();  // previous iteration finished with sQ / sdO / sdS / s_lse
      load_tile<D, 128>(sQ, qb, ldq, m0, len);
      load_tile<D, 128>(sdO, dob, lddo, m0, len);
      cp_async_commit();
      if (threadIdx.x < 64) {
        const int r = m0 + threadIdx.x;
        s_lse[threadIdx.x] = r < len ? lse[static_cast<int64_t>(h) * T + s0 + r] * LOG2E : 0.f;
        s_delta[threadIdx.x] = r < len ? delta[static_cast<int64_t>(h) * T + s0 + r] : 0.f;
      }
      cp_async_wait<0>();
      __syncthreads();

      const bool need_mask = (mt == nt) || (m0 + BM > len) || (n0 + BN > len);
      // two halves of 32 q columns keep the live register set below the 255 limit
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const int qc0 = half * 32;
        float st[4][4], dpt[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int e = 0; e < 4; ++e) st[i][e] = dpt[i][e] = 0.f;
#pragma unroll
        for (int kk = 0; kk < D / 16; ++kk) {
          uint32_t ka[4], va[4];
          ld_A<D>(ka, sK, warp * 16, kk * 16, lane);
          ld_A<D>(va, sV, warp * 16, kk * 16, lane);
#pragma unroll
          for (int np = 0; np < 2; ++np) {
            uint32_t b[4];
            ld_B_nk<D>(b, sQ, qc0 + np * 16, kk * 16, lane);
            mma16816(st[2 * np], ka, b[0], b[1]);
            mma16816(st[2 * np + 1], ka, b[2], b[3]);
            ld_B_nk<D>(b, sdO, qc0 + np * 16, kk * 16, lane);
            mma16816(dpt[2 * np], va, b[0], b[1]);
            mma16816(dpt[2 * np + 1], va, b[2], b[3]);
          }
        }
        uint32_t pa[2][4], dsa[2][4];  // bf16 A fragments: [k-step of 16 q][4]
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float p[4], ds[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int qc = qc0 + i * 8 + ((lane & 3) << 1) + (e & 1);  // q column within the tile
            const int kv = kv_lo + ((e >> 1) << 3);
            float pv = exp2f(st[i][e] * scale_log2 - s_lse[qc]);
            if (need_mask && ((m0 + qc) < kv || (m0 + qc) >= len || kv >= len)) pv = 0.f;
            p[e] = pv;
            ds[e] = pv * (dpt[i][e] - s_delta[qc]);
          }
          pa[i >> 1][(i & 1) * 2 + 0] = pack_bf16x2(p[0], p[1]);
          pa[i >> 1][(i & 1) * 2 + 1] = pack_bf16x2(p[2], p[3]);
          dsa[i >> 1][(i & 1) * 2 + 0] = pack_bf16x2(ds[0], ds[1]);
          dsa[i >> 1][(i & 1) * 2 + 1] = pack_bf16x2(ds[2], ds[3]);
          // dS^T tile in smem: [kv row][q col], 128B rows, 16B chunks swizzled by (row & 7)
#pragma unroll
          for (int hrow = 0; hrow < 2; ++hrow) {
            const int r = warp * 16 + (lane >> 2) + hrow * 8;
            const int chunk = (qc0 >> 3) + i;
            const uint32_t addr = sdS + r * 128 + ((chunk ^ (r & 7)) << 4) + ((lane & 3) << 2);
            const uint32_t val = pack_bf16x2(ds[2 * hrow], ds[2 * hrow + 1]);
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(val) : "memory");
          }
        }
        // dV += P^T dO ; dK += dS^T Q   (k dimension = these 32 q rows)
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) {
#pragma unroll
          for (int np = 0; np < D / 16; ++np) {
            uint32_t b[4];
            ld_B_kn<D>(b, sdO, qc0 + kk * 16, np * 16, lane);
            mma16816(dv_acc[2 * np], pa[kk], b[0], b[1]);
            mma16816(dv_acc[2 * np + 1], pa[kk], b[2], b[3]);
            ld_B_kn<D>(b, sQ, qc0 + kk * 16, np * 16, lane);
            mma16816(dk_acc[2 * np], dsa[kk], b[0], b[1]);
            mma16816(dk_acc[2 * np + 1], dsa[kk], b[2], b[3]);
          }
        }
      }
      __syncthreads();  // dS^T complete in smem
      // dQ[16 q rows of this warp, D] = dS[q, kv] K[kv, D];  A from the transposed dS^T tile
      {
        float dq[D / 8][4];
#pragma unroll
        for (int i = 0; i < D / 8; ++i)
#pragma unroll
          for (int e = 0; e < 4; ++e) dq[i][e] = 0.f;
#pragma unroll
        for (int kk = 0; kk < BN / 16; ++kk) {
          uint32_t a[4];
          ld_A_km<64>(a, sdS, warp * 16, kk * 16, lane);
#pragma unroll
          for (int np = 0; np < D / 16; ++np) {
            uint32_t b[4];
            ld_B_kn<D>(b, sK, kk * 16, np * 16, lane);
            mma16816(dq[2 * np], a, b[0], b[1]);
            mma16816(dq[2 * np + 1], a, b[2], b[3]);
          }
        }
#pragma unroll
        for (int hrow = 0; hrow < 2; ++hrow) {
          const int r = m0 + warp * 16 + (lane >> 2) + hrow * 8;
          if (r < len) {
            float* dst = dq_acc + static_cast<int64_t>(s0 + r) * lddq + h * D + ((lane & 3) << 1);
#pragma unroll
            for (int i = 0; i < D / 8; ++i) atomicAdd(reinterpret_cast<float2*>(dst + i * 8), make_float2(dq[i][2 * hrow], dq[i][2 * hrow + 1]));
          }
        }
      }
    }
  }
  // write dK (scaled) and dV for this kv tile / kv head
#pragma unroll
  for (int hrow = 0; hrow < 2; ++hrow) {
    const int r = kv_lo + hrow * 8;
    if (r < len) {
      __nv_bfloat16* dkr = dk + static_cast<int64_t>(s0 + r) * lddk + hk * D + ((lane & 3) << 1);
      __nv_bfloat16* dvr = dv + static_cast<int64_t>(s0 + r) * lddv + hk * D + ((lane & 3) << 1);
#pragma unroll
      for (int i = 0; i < D / 8; ++i) {
        *reinterpret_cast<uint32_t*>(dkr + i * 8) = pack_bf16x2(dk_acc[i][2 * hrow] * scale, dk_acc[i][2 * hrow + 1] * scale);
        *reinterpret_cast<uint32_t*>(dvr + i * 8) = pack_bf16x2(dv_acc[i][2 * hrow], dv_acc[i][2 * hrow + 1]);
      }
    }
  }
}

// dq (bf16, strided) = scale * dq_acc (fp32)
__global__ void __launch_bounds__(256) attn_dq_convert_kernel(const float* __restrict__ acc, __nv_bfloat16* __restrict__ dq, int64_t T,
                                                             int cols, int64_t ld_acc, int64_t lddq, float scale, int nbuf) {
  const int vpr = cols / 4;
  const int64_t total = T * vpr;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t t = i / vpr;
    const int c = static_cast<int>(i - t * vpr);
    float4 a = *reinterpret_cast<const float4*>(acc + t * ld_acc + c * 4);
    for (int b = 1; b < nbuf; ++b) {  // further accumulators (one per CTA, T rows each), summed in a fixed order
      const float4 x = *reinterpret_cast<const float4*>(acc + (b * T + t) * ld_acc + c * 4);
      a.x += x.x; a.y += x.y; a.z += x.z; a.w += x.w;
    }
    uint2 o;
    o.x = pack_bf16x2(a.x * scale, a.y * scale);
    o.y = pack_bf16x2(a.z * scale, a.w * scale);
    *reinterpret_cast<uint2*>(dq + t * lddq + c * 4) = o;
  }
}

// ------------------------------------------------------------------------------------------------ host
int attn_delta_launch(const void* o, const void* dout, float* delta, int64_t ldo, int64_t lddo, int Hq, int D, int T, cudaStream_t st) {
  const int64_t threads = static_cast<int64_t>(T) * Hq * (D / 8);
  attn_delta_kernel<<<static_cast<int>((threads + 255) / 256), 256, 0, st>>>(static_cast<const __nv_bfloat16*>(o),
                                                                                static_cast<const __nv_bfloat16*>(dout), delta, ldo, lddo, Hq, D, T);
  B200_CHECK_LAUNCH("attn_delta");
  return 0;
}
int attn_dq_convert_launch(const float* acc, int nbuf, void* dq, int64_t T, int cols, int64_t lddq, float scale, cudaStream_t st) {
  const int64_t total = T * (cols / 4);
  int blocks = static_cast<int>((total + 255) / 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  attn_dq_convert_kernel<<<blocks, 256, 0, st>>>(acc, static_cast<__nv_bfloat16*>(dq), T, cols, cols, lddq, scale, nbuf);
  B200_CHECK_LAUNCH("attn_dq_convert");
  return 0;
}

template <int D>
static int attn_fwd_launch(const void* q, const void* k, const void* v, void* o, float* lse, const int* cu, int nseq, int max_len,
                           int64_t ldq, int64_t ldk, int64_t ldv, int64_t ldo, int Hq, int Hkv, int T, float scale, cudaStream_t st) {
  constexpr int SMEM = 3 * 64 * D * 2;
  auto kern = attn_fwd_kernel<D>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
    if (e != cudaSuccess) return set_error(B200_ERR_CUDA, "attn_fwd smem attr: %s", cudaGetErrorString(e));
    configured = true;
  }
  dim3 grid((max_len + 63) / 64, Hq, nseq);
  kern<<<grid, 128, SMEM, st>>>(static_cast<const __nv_bfloat16*>(q), static_cast<const __nv_bfloat16*>(k),
                                static_cast<const __nv_bfloat16*>(v), static_cast<__nv_bfloat16*>(o), lse, cu, ldq, ldk, ldv, ldo, Hq,
                                Hkv, T, scale * 1.4426950408889634f);
  B200_CHECK_LAUNCH("attn_fwd");
  return 0;
}

int attn_fwd(const void* q, const void* k, const void* v, void* o, float* lse, const int* cu_seqlens, int nseq, int max_len,
             int64_t ldq, int64_t ldk, int64_t ldv, int64_t ldo, int Hq, int Hkv, int D, int T, float scale, cudaStream_t st) {
  if (Hq % Hkv) return set_error(B200_ERR_ARG, "attn: Hq %% Hkv != 0");
  if ((ldq | ldk | ldv | ldo) % 8) return set_error(B200_ERR_ARG, "attn: row pitches must be multiples of 8 elements");
  if (D == 128) return attn_fwd_launch<128>(q, k, v, o, lse, cu_seqlens, nseq, max_len, ldq, ldk, ldv, ldo, Hq, Hkv, T, scale, st);
  if (D == 64) return attn_fwd_launch<64>(q, k, v, o, lse, cu_seqlens, nseq, max_len, ldq, ldk, ldv, ldo, Hq, Hkv, T, scale, st);
  return set_error(B200_ERR_UNSUPPORTED, "attn: head_dim %d not in {64,128}", D);
}

size_t attn_bwd_workspace_bytes(int T, int Hq, int D, int max_seqlen) {
  // fp32 dQ accumulator + delta; a second accumulator when no sequence is longer than 512 tokens (attn_bwd_tc: bit-reproducible dQ)
  const size_t acc = static_cast<size_t>(T) * Hq * D * sizeof(float);
  return (max_seqlen <= 512 ? 2 : 1) * acc + static_cast<size_t>(T) * Hq * sizeof(float);
}

template <int D>
static int attn_bwd_launch(const void* q, const void* k, const void* v, const void* o, const void* dout, const float* lse, void* dq,
                           void* dk, void* dv, void* ws, const int* cu, int nseq, int max_len, int64_t ldq, int64_t ldk, int64_t ldv,
                           int64_t ldo, int64_t lddo, int64_t lddq, int64_t lddk, int64_t lddv, int Hq, int Hkv, int T, float scale,
                           cudaStream_t st) {
  constexpr int SMEM = 4 * 64 * D * 2 + 64 * 64 * 2 + 2 * 64 * 4;
  auto kern = attn_bwd_kernel<D>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
    if (e != cudaSuccess) return set_error(B200_ERR_CUDA, "attn_bwd smem attr: %s", cudaGetErrorString(e));
    configured = true;
  }
  float* dq_acc = static_cast<float*>(ws);
  float* delta = dq_acc + static_cast<size_t>(T) * Hq * D;
  cudaError_t e = cudaMemsetAsync(dq_acc, 0, static_cast<size_t>(T) * Hq * D * sizeof(float), st);
  if (e != cudaSuccess) return set_error(B200_ERR_CUDA, "attn_bwd memset: %s", cudaGetErrorString(e));
  if (int rc = attn_delta_launch(o, dout, delta, ldo, lddo, Hq, D, T, st)) return rc;
  dim3 grid((max_len + 63) / 64, Hkv, nseq);
  kern<<<grid, 128, SMEM, st>>>(static_cast<const __nv_bfloat16*>(q), static_cast<const __nv_bfloat16*>(k),
                                static_cast<const __nv_bfloat16*>(v), static_cast<const __nv_bfloat16*>(dout), lse, delta, dq_acc,
                                static_cast<__nv_bfloat16*>(dk), static_cast<__nv_bfloat16*>(dv), cu, ldq, ldk, ldv, lddo,
                                static_cast<int64_t>(Hq) * D, lddk, lddv, Hq, Hkv, T, scale, scale * 1.4426950408889634f);
  B200_CHECK_LAUNCH("attn_bwd");
  {
    const int cols = Hq * D;
    const int64_t total = static_cast<int64_t>(T) * (cols / 4);
    int blocks = static_cast<int>((total + 255) / 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    attn_dq_convert_kernel<<<blocks, 256, 0, st>>>(dq_acc, static_cast<__nv_bfloat16*>(dq), T, cols, cols, lddq, scale, 1);
    B200_CHECK_LAUNCH("attn_dq_convert");
  }
  return 0;
}

int attn_bwd(const void* q, const void* k, const void* v, const void* o, const void* dout, const float* lse, void* dq, void* dk,
             void* dv, void* ws, size_t ws_bytes, const int* cu_seqlens, int nseq, int max_len, int64_t ldq, int64_t ldk, int64_t ldv,
             int64_t ldo, int64_t lddo, int64_t lddq, int64_t lddk, int64_t lddv, int Hq, int Hkv, int D, int T, float scale, cudaStream_t st) {
  if (Hq % Hkv) return set_error(B200_ERR_ARG, "attn: Hq %% Hkv != 0");
  if (ws_bytes < static_cast<size_t>(T) * Hq * (D + 1) * sizeof(float)) return set_error(B200_ERR_ARG, "attn_bwd: workspace of %zu bytes is too small", ws_bytes);
  if ((ldq | ldk | ldv | ldo | lddo | lddq | lddk | lddv) % 8) return set_error(B200_ERR_ARG, "attn: row pitches must be multiples of 8 elements");
  if (D == 128)
    return attn_bwd_launch<128>(q, k, v, o, dout, lse, dq, dk, dv, ws, cu_seqlens, nseq, max_len, ldq, ldk, ldv, ldo, lddo, lddq, lddk,
                                lddv, Hq, Hkv, T, scale, st);
  if (D == 64)
    return attn_bwd_launch<64>(q, k, v, o, dout, lse, dq, dk, dv, ws, cu_seqlens, nseq, max_len, ldq, ldk, ldv, ldo, lddo, lddq, lddk,
                               lddv, Hq, Hkv, T, scale, st);
  return set_error(B200_ERR_UNSUPPORTED, "attn: head_dim %d not in {64,128}", D);
}

}  // namespace b200
