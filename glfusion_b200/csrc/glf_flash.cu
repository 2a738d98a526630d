// glf_flash.cu — mode='embedded' (softmax) attention of TPAVIModule (R/models/ours.py:878-902 with
// f_div_C = softmax(f, dim=-1)):   Y_b = softmax(Theta_b Phi_b^T) G_b      (no 1/sqrt(d) scale in the reference).
//
// Odd-width path (this header): exact attention with the N x N score matrix materialised for a bounded CHUNK of sequences
// at a time (scratch sized by attn_chunk()), every product on the tcgen05 GEMM of glf_gemm.cu:
//   fwd : S = Theta Phi^T (fp32) -> row softmax (P bf16, lse fp32) -> Y = P G
//   bwd : recompute S ; dPm = dY G^T ; P = exp(S - lse) ; dS = P o (dPm - delta) ; delta = rowsum(dY o Y)
//         dTheta = dS Phi ; dPhi = dS^T Theta ; dG = P^T dY        (transposes are MN-major operand reads, no copies)
// Memory is O(chunk * N^2), independent of the batch size; HBM traffic is O(N^2) per sequence, which is what a
// single-kernel flash version (scores kept in TMEM, online softmax in registers) removes — same entry points.

#include "glf_internal.h"
#include "glf_ptx.cuh"

namespace glf {

namespace {

__device__ __forceinline__ float block_reduce_max(float v, float* sm) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = blockDim.x >> 5;
  if (l == 0) sm[w] = v;
  __syncthreads();
  float r = sm[0];
  for (int i = 1; i < nw; ++i) r = fmaxf(r, sm[i]);
  __syncthreads();
  return r;
}
__device__ __forceinline__ float block_reduce_sum(float v, float* sm) {
  v = warp_sum(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = blockDim.x >> 5;
  if (l == 0) sm[w] = v;
  __syncthreads();
  float r = 0.f;
  for (int i = 0; i < nw; ++i) r += sm[i];
  __syncthreads();
  return r;
}

// one block per score row: P = softmax(S) in bf16 (padding columns [N, ld) zeroed), lse = max + log(sum)
__global__ void __launch_bounds__(256)
    softmax_rows_kernel(const float* __restrict__ S, bf16* __restrict__ P, float* __restrict__ lse, int N, int ld) {
  __shared__ float sm[8];
  const long long row = blockIdx.x;
  const float* s = S + row * ld;
  bf16* p = P + row * ld;
  float m = -INFINITY;
  for (int j = threadIdx.x; j < N; j += blockDim.x) m = fmaxf(m, s[j]);
  m = block_reduce_max(m, sm);
  float sum = 0.f;
  for (int j = threadIdx.x; j < N; j += blockDim.x) sum += __expf(s[j] - m);
  sum = block_reduce_sum(sum, sm);
  const float inv = 1.f / sum;
  for (int j = threadIdx.x; j < ld; j += blockDim.x) p[j] = __float2bfloat16(j < N ? __expf(s[j] - m) * inv : 0.f);
  if (threadIdx.x == 0) lse[row] = m + __logf(sum);
}

// delta[row] = sum_j dY[row, j] * Y[row, j]     (one warp per row)
__global__ void rowdot_kernel(const bf16* __restrict__ A, const bf16* __restrict__ B, float* __restrict__ out,
                              long long rows, int d) {
  const long long row = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float acc = 0.f;
  for (int j = lane * 2; j < d; j += 64) {
    const float2 a = unpack_bf16(*reinterpret_cast<const uint32_t*>(A + row * d + j));
    const float2 b = unpack_bf16(*reinterpret_cast<const uint32_t*>(B + row * d + j));
    acc = fmaf(a.x, b.x, fmaf(a.y, b.y, acc));
  }
  acc = warp_sum(acc);
  if (lane == 0) out[row] = acc;
}

// P = exp(S - lse[row]) ; dS = P * (dPm - delta[row]) ; both bf16, padding columns zeroed.  grid.y = row
__global__ void __launch_bounds__(256)
    softmax_bwd_kernel(const float* __restrict__ S, const float* __restrict__ dPm, const float* __restrict__ lse,
                       const float* __restrict__ delta, bf16* __restrict__ P, bf16* __restrict__ dS, int N, int ld) {
  const long long row = blockIdx.y;
  const float l = lse[row], dl = delta[row];
  const long long off = row * ld;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < ld; j += gridDim.x * blockDim.x) {
    float p = 0.f, ds = 0.f;
    if (j < N) {
      p = __expf(S[off + j] - l);
      ds = p * (dPm[off + j] - dl);
    }
    P[off + j] = __float2bfloat16(p);
    dS[off + j] = __float2bfloat16(ds);
  }
}


}  // namespace

// ------------------------------------------------------------------------------------------------ flash kernels
// Shared conventions of the three kernels below (all sm_100a, one CTA per SM, 320 threads):
//   warp 0        TMA producer (cp.async.bulk.tensor, SWIZZLE_128B tiles, mbarrier completion)
//   warp 1        MMA issuer   (one elected lane issues every tcgen05.mma; tcgen05.commit publishes results)
//   warps 2..5    compute warpgroup 0, warps 6..9 compute warpgroup 1: one TMEM lane (= one tile row) per thread;
//                 a warp may only touch TMEM lanes 32*(warp%4)..+31, so each group of four consecutive warps covers
//                 all 128 lanes.
// Scores / probabilities never leave the SM: S is accumulated in TMEM, read with tcgen05.ld, turned into bf16 P (or
// dS) in registers and written back over the consumed score columns with tcgen05.st, from where it is the A operand
// of the next tcgen05.mma (A-from-TMEM form).  exp() is one MUFU.EX2 per element on log2-scaled scores.
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

// ------------------------------------------------------------------------------------------------ flash forward
// One CTA = TWO 128-query tiles of one sequence (256 queries); it streams 128-key tiles of K = Phi and V = G.
// The two query tiles ping-pong: while warpgroup t does the softmax of S_t, the tensor pipe computes the other
// tile's P V product and next scores.  MMA issue order per key tile j (t = 0, 1):
//       wait P_t(j) ;  O_t += P_t(j) V_j ;  S_t(j+1) = Q_t K_{j+1}^T
// TMEM (512 columns): S0/P0 [0,128), S1/P1 [128,256), O0 [256,256+DV), O1 [384,384+DV).
// Online softmax with a lazy reference maximum (log2 domain): the running maximum is only raised -- and O rescaled in
// TMEM -- when a tile's maximum exceeds it by more than 8 (P <= 2^8 stays exact enough in bf16/fp32), so after the
// first few tiles the rescale pass disappears.  lse = (m + log2 l) ln 2 is exact irrespective of the reference.
// DQK: width of Q and K (the score product's K extent); DV: width of V, O, dY and dV.  mode='embedded' runs DQK = DV =
// Ci; mode='gaussian' reads Q = K = X (DQK = C) against V = G (DV = C').
template <int DQK, int DV>
struct FlashCfg {
  static constexpr uint32_t TILE_QK = 128 * DQK * 2;         // bytes of a 128 x DQK bf16 tile (DQK/64 swizzle atoms)
  static constexpr uint32_t TILE_V = 128 * DV * 2;
  static constexpr uint32_t SUB_QK = 64 * DQK * 2;           // bytes of a 64-row sub-tile
  static constexpr uint32_t SUB_V = 64 * DV * 2;
  static constexpr uint32_t SMEM_FWD = TILE_QK * 4 + TILE_V * 2 + 1024;   // 2 Q + 2 K + 2 V
  // 2 resident tiles (Q | dY, or K | V) + 4-deep ring of sub-tile pairs (K | V, or Q | dY)
  static constexpr uint32_t SMEM_BWD = TILE_QK + TILE_V + 4 * (SUB_QK + SUB_V) + 1024;
  static_assert(DQK % 64 == 0 && DV % 64 == 0 && DQK <= 128 && DV <= 128, "TMEM / shared-memory layout of the kernels");
};
constexpr int FLASH_THREADS = 320;

template <int DQK, int DV>
__global__ void __launch_bounds__(FLASH_THREADS, 1)
    flash_fwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                     const __grid_constant__ CUtensorMap tmV, bf16* __restrict__ Y, float* __restrict__ lse, int N,
                     int q_pairs) {
  using Cfg = FlashCfg<DQK, DV>;
  extern __shared__ uint8_t fsm_raw[];
  __shared__ uint64_t q_full, k_full[2], k_empty[2], v_full[2], v_empty[2], s_full[2], p_full[2], o_done[2];
  __shared__ uint32_t tmem_holder;
  const uint32_t base = (smem_u32(fsm_raw) + 1023u) & ~1023u;
  const uint32_t sQ = base, sK = base + 2 * Cfg::TILE_QK, sV = base + 4 * Cfg::TILE_QK;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x / q_pairs, qp = blockIdx.x % q_pairs;
  const int q0 = qp * 256;
  const int T = (N + 127) / 128;
  const int ntile = (q0 + 128 < N) ? 2 : 1;      // the last CTA of a sequence may own a single query tile

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    mbar_init(smem_u32(&q_full), 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&k_full[i]), 1);
      mbar_init(smem_u32(&k_empty[i]), 1);
      mbar_init(smem_u32(&v_full[i]), 1);
      mbar_init(smem_u32(&v_empty[i]), 1);
      mbar_init(smem_u32(&s_full[i]), 1);
      mbar_init(smem_u32(&p_full[i]), 128);
      mbar_init(smem_u32(&o_done[i]), 1);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_holder), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_holder;

  if (warp == 0) {
    if (elect_one()) {
      mbar_expect_tx(smem_u32(&q_full), ntile * Cfg::TILE_QK);
      for (int t = 0; t < ntile; ++t) {
#pragma unroll
        for (int kb = 0; kb < DQK / 64; ++kb)
          tma_load_4d(&tmQ, smem_u32(&q_full), sQ + t * Cfg::TILE_QK + kb * 16384, kb * 64, q0 + t * 128, b, 0);
      }
      for (int j = 0; j < T; ++j) {
        const int st = j & 1;
        const uint32_t ph = static_cast<uint32_t>(j >> 1) & 1u;
        mbar_wait(smem_u32(&k_empty[st]), ph ^ 1u);
        mbar_expect_tx(smem_u32(&k_full[st]), Cfg::TILE_QK);
#pragma unroll
        for (int kb = 0; kb < DQK / 64; ++kb)
          tma_load_4d(&tmK, smem_u32(&k_full[st]), sK + st * Cfg::TILE_QK + kb * 16384, kb * 64, j * 128, b, 0);
        mbar_wait(smem_u32(&v_empty[st]), ph ^ 1u);
        mbar_expect_tx(smem_u32(&v_full[st]), Cfg::TILE_V);
#pragma unroll
        for (int kb = 0; kb < DV / 64; ++kb)
          tma_load_4d(&tmV, smem_u32(&v_full[st]), sV + st * Cfg::TILE_V + kb * 16384, kb * 64, j * 128, b, 0);
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc_qk = make_idesc_bf16(128, 128, false, false);   // S = Q K^T : both K-major
      constexpr uint32_t idesc_pv = make_idesc_bf16(128, DV, false, true);     // O += P V  : A in TMEM, B MN-major
      auto issue_s = [&](int t, int j) {
        const uint32_t kbase = sK + (j & 1) * Cfg::TILE_QK;
        const uint32_t qbase = sQ + t * Cfg::TILE_QK;
#pragma unroll
        for (int k = 0; k < DQK / 16; ++k) {
          const uint32_t off = (k >> 2) * 16384 + (k & 3) * 32;
          umma_f16(tmem + t * 128, make_sdesc(qbase + off, 16, 1024), make_sdesc(kbase + off, 16, 1024), idesc_qk,
                   k != 0 ? 1u : 0u);
        }
        umma_commit(smem_u32(&s_full[t]));
      };
      mbar_wait(smem_u32(&q_full), 0);
      mbar_wait(smem_u32(&k_full[0]), 0);
      tc_fence_after();
      for (int t = 0; t < ntile; ++t) issue_s(t, 0);
      umma_commit(smem_u32(&k_empty[0]));
      for (int j = 0; j < T; ++j) {
        const int st = j & 1;
        const uint32_t ph = static_cast<uint32_t>(j >> 1) & 1u;
        const bool more = j + 1 < T;
        mbar_wait(smem_u32(&v_full[st]), ph);
        if (more) mbar_wait(smem_u32(&k_full[(j + 1) & 1]), static_cast<uint32_t>((j + 1) >> 1) & 1u);
        const uint32_t vbase = sV + st * Cfg::TILE_V;
        for (int t = 0; t < ntile; ++t) {
          mbar_wait(smem_u32(&p_full[t]), static_cast<uint32_t>(j) & 1u);   // P_t(j) is in TMEM, O_t rescaled
          tc_fence_after();
#pragma unroll
          for (int k = 0; k < 8; ++k)
            umma_f16_ts(tmem + 256 + t * 128, tmem + t * 128 + k * 8, make_sdesc(vbase + k * 2048, 16384, 1024),
                        idesc_pv, (j | k) != 0 ? 1u : 0u);
          umma_commit(smem_u32(&o_done[t]));
          if (more) issue_s(t, j + 1);           // overwrites P_t(j): ordered behind the product that reads it
        }
        umma_commit(smem_u32(&v_empty[st]));
        if (more) umma_commit(smem_u32(&k_empty[(j + 1) & 1]));
      }
    }
  } else {
    const int t = (warp - 2) >> 2;
    if (t < ntile) {
      const int q = warp & 3;
      const int row = q * 32 + lane;
      const uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
      const uint32_t scol = tmem + lane_addr + t * 128;
      const uint32_t ocol = tmem + lane_addr + 256 + t * 128;
      float m_run = -INFINITY;                   // reference maximum, log2 domain
      float l0 = 0.f, l1 = 0.f, l2 = 0.f, l3 = 0.f;
      for (int j = 0; j < T; ++j) {
        mbar_wait(smem_u32(&s_full[t]), static_cast<uint32_t>(j) & 1u);
        tc_fence_after();
        uint32_t s[4][32];
        tmem_ld_32x32(scol, s[0]);
        tmem_ld_32x32(scol + 32, s[1]);
        tmem_ld_32x32(scol + 64, s[2]);
        tmem_ld_32x32(scol + 96, s[3]);
        tmem_ld_wait();
        const int kv = N - j * 128;              // valid keys in this tile (>= 128 except for the last one)
        if (kv < 128) {
#pragma unroll
          for (int i = 0; i < 128; ++i)
            if (i >= kv) s[i >> 5][i & 31] = 0xff800000u;     // -inf
        }
        float x0 = __uint_as_float(s[0][0]), x1 = __uint_as_float(s[0][1]), x2 = __uint_as_float(s[0][2]),
              x3 = __uint_as_float(s[0][3]);
#pragma unroll
        for (int i = 4; i < 128; i += 4) {
          x0 = fmaxf(x0, __uint_as_float(s[i >> 5][i & 31]));
          x1 = fmaxf(x1, __uint_as_float(s[i >> 5][(i & 31) + 1]));
          x2 = fmaxf(x2, __uint_as_float(s[i >> 5][(i & 31) + 2]));
          x3 = fmaxf(x3, __uint_as_float(s[i >> 5][(i & 31) + 3]));
        }
        const float mx2 = fmaxf(fmaxf(x0, x1), fmaxf(x2, x3)) * kLog2e;
        if (__any_sync(0xffffffffu, mx2 > m_run + 8.f)) {
          const float m_new = fmaxf(m_run, mx2);
          const float alpha = ex2_approx(m_run - m_new);   // 0 on the first tile (m_run = -inf), 1 if unchanged
          if (j > 0) {
            mbar_wait(smem_u32(&o_done[t]), static_cast<uint32_t>(j - 1) & 1u);   // P(j-1) V(j-1) has landed in O
            tc_fence_after();
#pragma unroll 1
            for (int c = 0; c < DV / 32; ++c) {
              uint32_t v[32];
              tmem_ld_32x32(ocol + c * 32, v);
              tmem_ld_wait();
              uint32_t lo[16], hi[16];
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                lo[i] = __float_as_uint(__uint_as_float(v[i]) * alpha);
                hi[i] = __float_as_uint(__uint_as_float(v[16 + i]) * alpha);
              }
              tmem_st_32x32_x16(ocol + c * 32, lo);
              tmem_st_32x32_x16(ocol + c * 32 + 16, hi);
            }
          }
          l0 *= alpha; l1 *= alpha; l2 *= alpha; l3 *= alpha;
          m_run = m_new;
        }
        const float nm = -m_run;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint32_t pk[16];
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            const float p0 = ex2_approx(fmaf(__uint_as_float(s[c][i]), kLog2e, nm));
            const float p1 = ex2_approx(fmaf(__uint_as_float(s[c][i + 1]), kLog2e, nm));
            const float p2 = ex2_approx(fmaf(__uint_as_float(s[c][i + 2]), kLog2e, nm));
            const float p3 = ex2_approx(fmaf(__uint_as_float(s[c][i + 3]), kLog2e, nm));
            l0 += p0; l1 += p1; l2 += p2; l3 += p3;
            pk[i >> 1] = pack_bf16(p0, p1);
            pk[(i >> 1) + 1] = pack_bf16(p2, p3);
          }
          tmem_st_32x32_x16(scol + c * 16, pk);
        }
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(smem_u32(&p_full[t]));
      }
      // epilogue: O / l -> Y, lse
      mbar_wait(smem_u32(&o_done[t]), static_cast<uint32_t>(T - 1) & 1u);
      tc_fence_after();
      const float l = (l0 + l1) + (l2 + l3);
      const float inv = 1.f / l;
      const int grow = q0 + t * 128 + row;
      bf16* yrow = Y + (static_cast<long long>(b) * N + grow) * DV;
#pragma unroll 1
      for (int c = 0; c < DV / 32; ++c) {
        uint32_t v[32];
        tmem_ld_32x32(ocol + c * 32, v);
        tmem_ld_wait();
        if (grow < N) {
#pragma unroll
          for (int i = 0; i < 32; i += 8) {
            uint4 pk = make_uint4(pack_bf16(__uint_as_float(v[i]) * inv, __uint_as_float(v[i + 1]) * inv),
                                  pack_bf16(__uint_as_float(v[i + 2]) * inv, __uint_as_float(v[i + 3]) * inv),
                                  pack_bf16(__uint_as_float(v[i + 4]) * inv, __uint_as_float(v[i + 5]) * inv),
                                  pack_bf16(__uint_as_float(v[i + 6]) * inv, __uint_as_float(v[i + 7]) * inv));
            *reinterpret_cast<uint4*>(yrow + c * 32 + i) = pk;
          }
        }
      }
      if (grow < N) lse[static_cast<long long>(b) * N + grow] = (m_run + log2f(l)) * kLn2;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

// ------------------------------------------------------------------------------------------------ flash backward
// Recompute-based (nothing N x N is stored): with lse from the forward and delta = rowsum(dY o Y),
//   P = exp(S - lse) ,  dS = P o (dY V^T - delta)
//   dQ kernel   (CTA = 128 queries, streams 64-key sub-tiles):  S = Q K^T, dP = dY V^T -> dS (bf16, TMEM) -> dQ += dS K
//   dK/dV kernel(CTA = 128 keys, streams 64-query sub-tiles):   S^T = K Q^T, dP^T = V dY^T -> P^T, dS^T (bf16, TMEM)
//                                                                -> dV += P^T dY , dK += dS^T Q
// Every product is a tcgen05.mma; P / dS never leave TMEM (they are the A operand of the second product); transposed
// uses of a tile (Q as [q,d] and as [d,q]) are the same shared-memory bytes read through K-major / MN-major descriptors.
// Deterministic: no atomics.  Scores are recomputed once per kernel (7 products per tile pair instead of 5).
// Pipelining: the 128 x 64 score / dP blocks are double-buffered in TMEM (stage = sub-tile parity) and the two compute
// warpgroups alternate sub-tiles, so the tensor pipe computes sub-tile j+1's scores and sub-tile j-1's accumulation
// while a warpgroup turns sub-tile j's scores into dS.
//   dQ kernel TMEM   : stage s at [128 s, 128 s + 128): S [0,64) (dS bf16 over [0,32)), dP [64,128);  dQ at [256, 256+DQK)
//   dK/dV kernel TMEM: dV [0,DV), dK [128,128+DQK); stage s at [256 + 128 s, ..): S^T [0,64) (P^T bf16 over [0,32)),
//                      dP^T [64,128) (dS^T bf16 over [64,96))
// dQ, dK and dV go to their own row-strided outputs (ld_* elements between rows).
template <int DQK, int DV>
__global__ void __launch_bounds__(FLASH_THREADS, 1)
    flash_bwd_dq_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                        const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmdY,
                        const float* __restrict__ lse, const float* __restrict__ delta, bf16* __restrict__ dQ,
                        long long ld_dq, int N, int q_tiles) {
  using Cfg = FlashCfg<DQK, DV>;
  constexpr int RING = 4;
  extern __shared__ uint8_t fsm_raw[];
  __shared__ uint64_t q_full, kv_full[RING], kv_empty[RING], s_full[2], ds_full[2], dq_done;
  __shared__ uint32_t tmem_holder;
  const uint32_t base = (smem_u32(fsm_raw) + 1023u) & ~1023u;
  const uint32_t sQ = base, sdY = base + Cfg::TILE_QK, sRing = sdY + Cfg::TILE_V;   // ring slot: K_sub | V_sub
  constexpr uint32_t SLOT = Cfg::SUB_QK + Cfg::SUB_V;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x / q_tiles, qt = blockIdx.x % q_tiles;
  const int q0 = qt * 128;
  const int T = (N + 63) / 64;       // 64-key sub-tiles
  constexpr uint32_t COL_DQ = 256;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmK); tma_prefetch_desc(&tmV); tma_prefetch_desc(&tmdY);
    mbar_init(smem_u32(&q_full), 1);
    for (int i = 0; i < RING; ++i) {
      mbar_init(smem_u32(&kv_full[i]), 1);
      mbar_init(smem_u32(&kv_empty[i]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&s_full[i]), 1);
      mbar_init(smem_u32(&ds_full[i]), 128);
    }
    mbar_init(smem_u32(&dq_done), 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_holder), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_holder;

  if (warp == 0) {
    if (elect_one()) {
      mbar_expect_tx(smem_u32(&q_full), Cfg::TILE_QK + Cfg::TILE_V);
#pragma unroll
      for (int kb = 0; kb < DQK / 64; ++kb) tma_load_4d(&tmQ, smem_u32(&q_full), sQ + kb * 16384, kb * 64, q0, b, 0);
#pragma unroll
      for (int kb = 0; kb < DV / 64; ++kb) tma_load_4d(&tmdY, smem_u32(&q_full), sdY + kb * 16384, kb * 64, q0, b, 0);
      for (int j = 0; j < T; ++j) {
        const int r = j % RING;
        const uint32_t ph = static_cast<uint32_t>(j / RING) & 1u;
        mbar_wait(smem_u32(&kv_empty[r]), ph ^ 1u);
        mbar_expect_tx(smem_u32(&kv_full[r]), SLOT);
        const uint32_t slot = sRing + r * SLOT;
#pragma unroll
        for (int kb = 0; kb < DQK / 64; ++kb)
          tma_load_4d(&tmK, smem_u32(&kv_full[r]), slot + kb * 8192, kb * 64, j * 64, b, 0);
#pragma unroll
        for (int kb = 0; kb < DV / 64; ++kb)
          tma_load_4d(&tmV, smem_u32(&kv_full[r]), slot + Cfg::SUB_QK + kb * 8192, kb * 64, j * 64, b, 0);
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc_s = make_idesc_bf16(128, 64, false, false);
      constexpr uint32_t idesc_dq = make_idesc_bf16(128, DQK, false, true);
      auto issue_sdp = [&](int j) {
        const int r = j % RING;
        mbar_wait(smem_u32(&kv_full[r]), static_cast<uint32_t>(j / RING) & 1u);
        tc_fence_after();
        const uint32_t kb_ = sRing + r * SLOT, vb_ = kb_ + Cfg::SUB_QK;
        const uint32_t stage = tmem + (j & 1) * 128;
#pragma unroll
        for (int k = 0; k < DQK / 16; ++k) {   // S = Q K_sub^T
          const uint32_t offa = (k >> 2) * 16384 + (k & 3) * 32, offb = (k >> 2) * 8192 + (k & 3) * 32;
          umma_f16(stage, make_sdesc(sQ + offa, 16, 1024), make_sdesc(kb_ + offb, 16, 1024), idesc_s, k != 0 ? 1u : 0u);
        }
#pragma unroll
        for (int k = 0; k < DV / 16; ++k) {   // dP = dY V_sub^T
          const uint32_t offa = (k >> 2) * 16384 + (k & 3) * 32, offb = (k >> 2) * 8192 + (k & 3) * 32;
          umma_f16(stage + 64, make_sdesc(sdY + offa, 16, 1024), make_sdesc(vb_ + offb, 16, 1024), idesc_s,
                   k != 0 ? 1u : 0u);
        }
        umma_commit(smem_u32(&s_full[j & 1]));
      };
      mbar_wait(smem_u32(&q_full), 0);
      tc_fence_after();
      issue_sdp(0);
      for (int j = 0; j < T; ++j) {
        const int r = j % RING;
        if (j + 1 < T) issue_sdp(j + 1);     // stage (j+1)&1 was drained by sub-tile j-1 (ordered behind its dQ product)
        mbar_wait(smem_u32(&ds_full[j & 1]), static_cast<uint32_t>(j >> 1) & 1u);   // dS (bf16) in stage columns [0,32)
        tc_fence_after();
        const uint32_t kb_ = sRing + r * SLOT;
#pragma unroll
        for (int k = 0; k < 4; ++k)          // dQ += dS K_sub   (A from TMEM, K sub-tile read MN-major)
          umma_f16_ts(tmem + COL_DQ, tmem + (j & 1) * 128 + k * 8, make_sdesc(kb_ + k * 2048, 8192, 1024), idesc_dq,
                      (j | k) != 0 ? 1u : 0u);
        umma_commit(smem_u32(&kv_empty[r]));
        if (j == T - 1) umma_commit(smem_u32(&dq_done));
      }
    }
  } else {
    const int wg = (warp - 2) >> 2;
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int grow = q0 + row;
    const uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
    const bool rvalid = grow < N;
    const float l2 = rvalid ? lse[static_cast<long long>(b) * N + grow] * kLog2e : 0.f;
    const float dl = rvalid ? delta[static_cast<long long>(b) * N + grow] : 0.f;
    const uint32_t stage = tmem + lane_addr + wg * 128;
    for (int j = wg; j < T; j += 2) {
      mbar_wait(smem_u32(&s_full[wg]), static_cast<uint32_t>(j >> 1) & 1u);
      tc_fence_after();
      uint32_t sv[2][32], dv[2][32];
      tmem_ld_32x32(stage, sv[0]);
      tmem_ld_32x32(stage + 32, sv[1]);
      tmem_ld_32x32(stage + 64, dv[0]);
      tmem_ld_32x32(stage + 96, dv[1]);
      tmem_ld_wait();
      const int kv = rvalid ? N - j * 64 : 0;   // valid keys of this sub-tile for this row (0: whole row is padding)
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t pk[16];
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          const int e = c * 32 + i;
          float d0 = ex2_approx(fmaf(__uint_as_float(sv[c][i]), kLog2e, -l2)) * (__uint_as_float(dv[c][i]) - dl);
          float d1 = ex2_approx(fmaf(__uint_as_float(sv[c][i + 1]), kLog2e, -l2)) * (__uint_as_float(dv[c][i + 1]) - dl);
          if (kv < 64) {
            if (e >= kv) d0 = 0.f;
            if (e + 1 >= kv) d1 = 0.f;
          }
          pk[i >> 1] = pack_bf16(d0, d1);
        }
        tmem_st_32x32_x16(stage + c * 16, pk);
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(smem_u32(&ds_full[wg]));
    }
    mbar_wait(smem_u32(&dq_done), 0);
    tc_fence_after();
    bf16* orow = dQ + (static_cast<long long>(b) * N + grow) * ld_dq;
    // the two warpgroups split the DQK columns of dQ
#pragma unroll 1
    for (int c = wg * (DQK / 64); c < (wg + 1) * (DQK / 64); ++c) {
      uint32_t v[32];
      tmem_ld_32x32(tmem + lane_addr + COL_DQ + c * 32, v);
      tmem_ld_wait();
      if (rvalid) {
#pragma unroll
        for (int i = 0; i < 32; i += 8) {
          uint4 pk = make_uint4(pack_bf16(__uint_as_float(v[i]), __uint_as_float(v[i + 1])),
                                pack_bf16(__uint_as_float(v[i + 2]), __uint_as_float(v[i + 3])),
                                pack_bf16(__uint_as_float(v[i + 4]), __uint_as_float(v[i + 5])),
                                pack_bf16(__uint_as_float(v[i + 6]), __uint_as_float(v[i + 7])));
          *reinterpret_cast<uint4*>(orow + c * 32 + i) = pk;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

template <int DQK, int DV>
__global__ void __launch_bounds__(FLASH_THREADS, 1)
    flash_bwd_dkv_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                         const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmdY,
                         const float* __restrict__ lse, const float* __restrict__ delta, bf16* __restrict__ dK,
                         long long ld_dk, bf16* __restrict__ dV, long long ld_dv, int N, int kv_tiles) {
  using Cfg = FlashCfg<DQK, DV>;
  constexpr int RING = 4;
  extern __shared__ uint8_t fsm_raw[];
  __shared__ uint64_t kv_full, q_full[RING], q_empty[RING], s_full[2], p_full[2], acc_done;
  __shared__ uint32_t tmem_holder;
  __shared__ __align__(16) float lse_sm[2][2][64], del_sm[2][2][64];   // [warpgroup][buffer][query of the sub-tile]
  const uint32_t base = (smem_u32(fsm_raw) + 1023u) & ~1023u;
  const uint32_t sK = base, sV = base + Cfg::TILE_QK, sRing = sV + Cfg::TILE_V;   // ring slot: Q_sub | dY_sub
  constexpr uint32_t SLOT = Cfg::SUB_QK + Cfg::SUB_V;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x / kv_tiles, kt = blockIdx.x % kv_tiles;
  const int k0 = kt * 128;
  const int T = (N + 63) / 64;   // 64-query sub-tiles
  constexpr uint32_t COL_DV = 0, COL_DK = 128, COL_ST = 256;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmK); tma_prefetch_desc(&tmV); tma_prefetch_desc(&tmdY);
    mbar_init(smem_u32(&kv_full), 1);
    for (int i = 0; i < RING; ++i) {
      mbar_init(smem_u32(&q_full[i]), 1);
      mbar_init(smem_u32(&q_empty[i]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&s_full[i]), 1);
      mbar_init(smem_u32(&p_full[i]), 128);
    }
    mbar_init(smem_u32(&acc_done), 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_holder), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_holder;

  if (warp == 0) {
    if (elect_one()) {
      mbar_expect_tx(smem_u32(&kv_full), Cfg::TILE_QK + Cfg::TILE_V);
#pragma unroll
      for (int kb = 0; kb < DQK / 64; ++kb) tma_load_4d(&tmK, smem_u32(&kv_full), sK + kb * 16384, kb * 64, k0, b, 0);
#pragma unroll
      for (int kb = 0; kb < DV / 64; ++kb) tma_load_4d(&tmV, smem_u32(&kv_full), sV + kb * 16384, kb * 64, k0, b, 0);
      for (int i = 0; i < T; ++i) {
        const int r = i % RING;
        const uint32_t ph = static_cast<uint32_t>(i / RING) & 1u;
        mbar_wait(smem_u32(&q_empty[r]), ph ^ 1u);
        mbar_expect_tx(smem_u32(&q_full[r]), SLOT);
        const uint32_t slot = sRing + r * SLOT;
#pragma unroll
        for (int kb = 0; kb < DQK / 64; ++kb)
          tma_load_4d(&tmQ, smem_u32(&q_full[r]), slot + kb * 8192, kb * 64, i * 64, b, 0);
#pragma unroll
        for (int kb = 0; kb < DV / 64; ++kb)
          tma_load_4d(&tmdY, smem_u32(&q_full[r]), slot + Cfg::SUB_QK + kb * 8192, kb * 64, i * 64, b, 0);
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc_s = make_idesc_bf16(128, 64, false, false);
      constexpr uint32_t idesc_dv = make_idesc_bf16(128, DV, false, true);
      constexpr uint32_t idesc_dk = make_idesc_bf16(128, DQK, false, true);
      auto issue_sdp = [&](int i) {
        const int r = i % RING;
        mbar_wait(smem_u32(&q_full[r]), static_cast<uint32_t>(i / RING) & 1u);
        tc_fence_after();
        const uint32_t qb_ = sRing + r * SLOT, yb_ = qb_ + Cfg::SUB_QK;
        const uint32_t stage = tmem + COL_ST + (i & 1) * 128;
#pragma unroll
        for (int k = 0; k < DQK / 16; ++k) {   // S^T = K Q_sub^T
          const uint32_t offa = (k >> 2) * 16384 + (k & 3) * 32, offb = (k >> 2) * 8192 + (k & 3) * 32;
          umma_f16(stage, make_sdesc(sK + offa, 16, 1024), make_sdesc(qb_ + offb, 16, 1024), idesc_s, k != 0 ? 1u : 0u);
        }
#pragma unroll
        for (int k = 0; k < DV / 16; ++k) {   // dP^T = V dY_sub^T
          const uint32_t offa = (k >> 2) * 16384 + (k & 3) * 32, offb = (k >> 2) * 8192 + (k & 3) * 32;
          umma_f16(stage + 64, make_sdesc(sV + offa, 16, 1024), make_sdesc(yb_ + offb, 16, 1024), idesc_s,
                   k != 0 ? 1u : 0u);
        }
        umma_commit(smem_u32(&s_full[i & 1]));
      };
      mbar_wait(smem_u32(&kv_full), 0);
      tc_fence_after();
      issue_sdp(0);
      for (int i = 0; i < T; ++i) {
        const int r = i % RING;
        if (i + 1 < T) issue_sdp(i + 1);
        mbar_wait(smem_u32(&p_full[i & 1]), static_cast<uint32_t>(i >> 1) & 1u);   // P^T [0,32), dS^T [64,96) (bf16)
        tc_fence_after();
        const uint32_t qb_ = sRing + r * SLOT, yb_ = qb_ + Cfg::SUB_QK;
        const uint32_t stage = tmem + COL_ST + (i & 1) * 128;
#pragma unroll
        for (int k = 0; k < 4; ++k)          // dV += P^T dY_sub   (dY sub-tile read MN-major)
          umma_f16_ts(tmem + COL_DV, stage + k * 8, make_sdesc(yb_ + k * 2048, 8192, 1024), idesc_dv,
                      (i | k) != 0 ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < 4; ++k)          // dK += dS^T Q_sub   (Q sub-tile read MN-major)
          umma_f16_ts(tmem + COL_DK, stage + 64 + k * 8, make_sdesc(qb_ + k * 2048, 8192, 1024), idesc_dk,
                      (i | k) != 0 ? 1u : 0u);
        umma_commit(smem_u32(&q_empty[r]));
        if (i == T - 1) umma_commit(smem_u32(&acc_done));
      }
    }
  } else {
    const int wg = (warp - 2) >> 2;
    const int q = warp & 3;
    const int row = q * 32 + lane;          // key row of this thread
    const int gkey = k0 + row;
    const bool kvalid = gkey < N;
    const uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
    const int e = ((warp - 2) & 3) * 32 + lane;   // 0..127 inside the warpgroup
    const uint32_t stage = tmem + lane_addr + COL_ST + wg * 128;
    int sb = 0;
    for (int i = wg; i < T; i += 2, sb ^= 1) {
      {  // per-query lse / delta of this sub-tile (columns of S^T): published to the warpgroup by a named barrier
        const int gq = i * 64 + (e & 63);
        const bool ok = gq < N;
        if (e < 64) lse_sm[wg][sb][e] = ok ? lse[static_cast<long long>(b) * N + gq] * kLog2e : 0.f;
        else del_sm[wg][sb][e - 64] = ok ? delta[static_cast<long long>(b) * N + gq] : 0.f;
      }
      named_bar_sync(1 + wg, 128);
      mbar_wait(smem_u32(&s_full[wg]), static_cast<uint32_t>(i >> 1) & 1u);
      tc_fence_after();
      uint32_t sv[2][32], dv[2][32];
      tmem_ld_32x32(stage, sv[0]);
      tmem_ld_32x32(stage + 32, sv[1]);
      tmem_ld_32x32(stage + 64, dv[0]);
      tmem_ld_32x32(stage + 96, dv[1]);
      tmem_ld_wait();
      const int qv = kvalid ? N - i * 64 : 0;   // valid queries of this sub-tile for this key row
      const float4* ls4 = reinterpret_cast<const float4*>(lse_sm[wg][sb]);
      const float4* dl4 = reinterpret_cast<const float4*>(del_sm[wg][sb]);
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t pp[16], pd[16];
#pragma unroll
        for (int t = 0; t < 32; t += 4) {
          const int col = c * 32 + t;
          const float4 L = ls4[col >> 2], Dl = dl4[col >> 2];
          float p0 = ex2_approx(fmaf(__uint_as_float(sv[c][t]), kLog2e, -L.x));
          float p1 = ex2_approx(fmaf(__uint_as_float(sv[c][t + 1]), kLog2e, -L.y));
          float p2 = ex2_approx(fmaf(__uint_as_float(sv[c][t + 2]), kLog2e, -L.z));
          float p3 = ex2_approx(fmaf(__uint_as_float(sv[c][t + 3]), kLog2e, -L.w));
          if (qv < 64) {
            if (col >= qv) p0 = 0.f;
            if (col + 1 >= qv) p1 = 0.f;
            if (col + 2 >= qv) p2 = 0.f;
            if (col + 3 >= qv) p3 = 0.f;
          }
          const float d0 = p0 * (__uint_as_float(dv[c][t]) - Dl.x);
          const float d1 = p1 * (__uint_as_float(dv[c][t + 1]) - Dl.y);
          const float d2 = p2 * (__uint_as_float(dv[c][t + 2]) - Dl.z);
          const float d3 = p3 * (__uint_as_float(dv[c][t + 3]) - Dl.w);
          pp[t >> 1] = pack_bf16(p0, p1);
          pp[(t >> 1) + 1] = pack_bf16(p2, p3);
          pd[t >> 1] = pack_bf16(d0, d1);
          pd[(t >> 1) + 1] = pack_bf16(d2, d3);
        }
        tmem_st_32x32_x16(stage + c * 16, pp);
        tmem_st_32x32_x16(stage + 64 + c * 16, pd);
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(smem_u32(&p_full[wg]));
    }
    mbar_wait(smem_u32(&acc_done), 0);
    tc_fence_after();
    // warpgroup 0 writes dK, warpgroup 1 writes dV
    bf16* orow = wg == 0 ? dK + (static_cast<long long>(b) * N + gkey) * ld_dk
                         : dV + (static_cast<long long>(b) * N + gkey) * ld_dv;
    const uint32_t acc = tmem + lane_addr + (wg == 0 ? COL_DK : COL_DV);
#pragma unroll 1
    for (int c = 0; c < (wg == 0 ? DQK : DV) / 32; ++c) {
      uint32_t v[32];
      tmem_ld_32x32(acc + c * 32, v);
      tmem_ld_wait();
      if (kvalid) {
#pragma unroll
        for (int t = 0; t < 32; t += 8) {
          uint4 a = make_uint4(pack_bf16(__uint_as_float(v[t]), __uint_as_float(v[t + 1])),
                               pack_bf16(__uint_as_float(v[t + 2]), __uint_as_float(v[t + 3])),
                               pack_bf16(__uint_as_float(v[t + 4]), __uint_as_float(v[t + 5])),
                               pack_bf16(__uint_as_float(v[t + 6]), __uint_as_float(v[t + 7])));
          *reinterpret_cast<uint4*>(orow + c * 32 + t) = a;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

// per-CTA partial column sums of a bf16 [rows, Ccols] matrix with row stride ld (bias gradients = column sums of dP):
// part [grid][2][Ccols]
__global__ void __launch_bounds__(256) colsum_bf16_kernel(const bf16* __restrict__ A, float* __restrict__ part,
                                                         long long rows, int Ccols, long long ld) {
  // thread = one 8-column group per pass; rows strided over (blockIdx, row lane)
  const int groups = Ccols / 8;
  for (int g0 = 0; g0 < groups; g0 += 64) {
    const int g = g0 + (threadIdx.x & 63);
    const int ty = threadIdx.x >> 6;
    float s[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) s[t] = 0.f;
    if (g < groups) {
      for (long long r = static_cast<long long>(blockIdx.x) * 4 + ty; r < rows; r += static_cast<long long>(gridDim.x) * 4) {
        const uint4 v = *reinterpret_cast<const uint4*>(A + r * ld + g * 8);
        const uint32_t* u = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const float2 x = unpack_bf16(u[t]);
          s[2 * t] += x.x;
          s[2 * t + 1] += x.y;
        }
      }
    }
    __shared__ float sm[4][64 * 8];
#pragma unroll
    for (int t = 0; t < 8; ++t) sm[ty][(threadIdx.x & 63) * 8 + t] = s[t];
    __syncthreads();
    for (int idx = threadIdx.x; idx < 64 * 8; idx += 256) {
      const int col = g0 * 8 + idx;
      if (col < Ccols)
        part[static_cast<long long>(blockIdx.x) * 2 * Ccols + col] = sm[0][idx] + sm[1][idx] + sm[2][idx] + sm[3][idx];
    }
    __syncthreads();
  }
}

template <int DQK, int DV>
static int launch_flash_bwd(const AttnArgs& a, const bf16* dY, const float* lse, const float* delta, int B, int N,
                            cudaStream_t stream) {
  using Cfg = FlashCfg<DQK, DV>;
  // 128-row boxes for the operand that stays resident in a CTA, 64-row boxes for the streamed sub-tiles
  CUtensorMap tq128, tk128, tv128, ty128, tq64, tk64, tv64, ty64;
  const long long n = N;
  int rc;
  if ((rc = make_tmap_bf16(&tq128, a.q, DQK, N, B, a.ldq, n * a.ldq, 128))) return rc;
  if ((rc = make_tmap_bf16(&tk128, a.k, DQK, N, B, a.ldk, n * a.ldk, 128))) return rc;
  if ((rc = make_tmap_bf16(&tv128, a.v, DV, N, B, a.ldv, n * a.ldv, 128))) return rc;
  if ((rc = make_tmap_bf16(&ty128, dY, DV, N, B, DV, n * DV, 128))) return rc;
  if ((rc = make_tmap_bf16(&tq64, a.q, DQK, N, B, a.ldq, n * a.ldq, 64))) return rc;
  if ((rc = make_tmap_bf16(&tk64, a.k, DQK, N, B, a.ldk, n * a.ldk, 64))) return rc;
  if ((rc = make_tmap_bf16(&tv64, a.v, DV, N, B, a.ldv, n * a.ldv, 64))) return rc;
  if ((rc = make_tmap_bf16(&ty64, dY, DV, N, B, DV, n * DV, 64))) return rc;
  const uint32_t smem = Cfg::SMEM_BWD;
  const int tiles = (N + 127) / 128;
  {
    auto kern = flash_bwd_dq_kernel<DQK, DV>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(flash_bwd_dq)");
    kern<<<B * tiles, FLASH_THREADS, smem, stream>>>(tq128, tk64, tv64, ty128, lse, delta, a.dq, a.ld_dq, N, tiles);
    if ((rc = check_cuda(cudaGetLastError(), "flash_bwd_dq launch"))) return rc;
  }
  {
    auto kern = flash_bwd_dkv_kernel<DQK, DV>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(flash_bwd_dkv)");
    kern<<<B * tiles, FLASH_THREADS, smem, stream>>>(tq64, tk128, tv128, ty64, lse, delta, a.dk, a.ld_dk, a.dvo,
                                                     a.ld_dv, N, tiles);
    if ((rc = check_cuda(cudaGetLastError(), "flash_bwd_dkv launch"))) return rc;
  }
  return 0;
}

template <int DQK, int DV>
static int launch_flash_fwd(const AttnArgs& a, bf16* Y, float* lse, int B, int N, cudaStream_t stream) {
  using Cfg = FlashCfg<DQK, DV>;
  CUtensorMap tq, tk, tv;
  const long long n = N;
  int rc;
  if ((rc = make_tmap_bf16(&tq, a.q, DQK, N, B, a.ldq, n * a.ldq, 128))) return rc;
  if ((rc = make_tmap_bf16(&tk, a.k, DQK, N, B, a.ldk, n * a.ldk, 128))) return rc;
  if ((rc = make_tmap_bf16(&tv, a.v, DV, N, B, a.ldv, n * a.ldv, 128))) return rc;
  auto kern = flash_fwd_kernel<DQK, DV>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_FWD);
  if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(flash_fwd)");
  const int q_pairs = (N + 255) / 256;
  kern<<<B * q_pairs, FLASH_THREADS, Cfg::SMEM_FWD, stream>>>(tq, tk, tv, Y, lse, N, q_pairs);
  return check_cuda(cudaGetLastError(), "flash_fwd launch");
}

int attn_ld(int N) { return (N + 7) & ~7; }

// sequences per chunk so that the backward scratch (12 bytes per score) stays under ~2 GiB (at least 1)
int attn_chunk(long long B, long long N) {
  const long long per_seq = static_cast<long long>(attn_ld(static_cast<int>(N))) * N * 12;
  long long nb = (2LL << 30) / (per_seq > 0 ? per_seq : 1);
  if (nb < 1) nb = 1;
  if (nb > B) nb = B;
  return static_cast<int>(nb);
}
size_t attn_scratch_bytes(long long B, long long N, bool backward) {
  const size_t nb = attn_chunk(B, N);
  const size_t per = static_cast<size_t>(attn_ld(static_cast<int>(N))) * N;
  return nb * per * (backward ? 12 : 6) + 1024;
}

AttnArgs attn_args_embedded(const bf16* P3, bf16* dP3, int Ci) {
  AttnArgs a;
  a.q = P3; a.k = P3 + Ci; a.v = P3 + 2 * Ci;
  a.ldq = a.ldk = a.ldv = 3LL * Ci;
  a.wqk = a.wv = Ci;
  a.dq = dP3; a.dk = dP3 ? dP3 + Ci : nullptr; a.dvo = dP3 ? dP3 + 2 * Ci : nullptr;
  a.ld_dq = a.ld_dk = a.ld_dv = 3LL * Ci;
  a.bias_qkv = true;
  return a;
}

AttnArgs attn_args_gaussian(const bf16* X, const bf16* G, bf16* dXa, bf16* dXb, bf16* dG, long long ld_dx,
                            long long ld_dg, int C, int Ci) {
  AttnArgs a;
  a.q = a.k = X;
  a.ldq = a.ldk = C;
  a.v = G; a.ldv = Ci;
  a.wqk = C; a.wv = Ci;
  a.dq = dXa; a.dk = dXb; a.dvo = dG;
  a.ld_dq = a.ld_dk = ld_dx; a.ld_dv = ld_dg;
  a.bias_qkv = false;
  return a;
}

bool attn_flash_supported(int wqk, int wv) {
  return (wqk == 64 && wv == 64) || (wqk == 128 && wv == 64) || (wqk == 128 && wv == 128);
}

static int attn_fwd_materialized(const AttnArgs& a, bf16* Y, float* lse, int B, int N, void* scratch,
                                 cudaStream_t stream) {
  const int ld = attn_ld(N);
  const int nb = attn_chunk(B, N);
  const size_t per = static_cast<size_t>(ld) * N;
  float* S = reinterpret_cast<float*>(scratch);
  bf16* Pm = reinterpret_cast<bf16*>(S + nb * per);
  const long long n = N;
  for (int b0 = 0; b0 < B; b0 += nb) {
    const int cb = (B - b0 < nb) ? (B - b0) : nb;
    const bf16* Qb = a.q + b0 * n * a.ldq;
    const bf16* Kb = a.k + b0 * n * a.ldk;
    const bf16* Vb = a.v + b0 * n * a.ldv;
    {  // S = Q K^T   (columns [N, ld) come out as zeros: K rows beyond N are TMA out-of-bounds)
      GemmArgs g;
      g.A = opnd(Qb, 0, a.ldq, n * a.ldq);
      g.B = opnd(Kb, 0, a.ldk, n * a.ldk);
      g.B.rows = N;
      g.M = N; g.N = ld; g.K = a.wqk; g.batch = cb;
      g.out_kind = 1;
      g.D = S; g.ldd = ld; g.strideD = static_cast<long long>(per);
      int rc = gemm(g, stream);
      if (rc) return rc;
    }
    softmax_rows_kernel<<<static_cast<unsigned>(static_cast<long long>(cb) * N), 256, 0, stream>>>(
        S, Pm, lse + static_cast<long long>(b0) * N, N, ld);
    int rc = check_cuda(cudaGetLastError(), "softmax_rows launch");
    if (rc) return rc;
    {  // Y = P V
      GemmArgs g;
      g.A = opnd(Pm, 0, ld, static_cast<long long>(per));
      g.B = opnd(Vb, 1, a.ldv, n * a.ldv);
      g.M = N; g.N = a.wv; g.K = N; g.batch = cb;
      g.D = Y + b0 * n * a.wv; g.ldd = a.wv; g.strideD = n * a.wv;
      rc = gemm(g, stream);
      if (rc) return rc;
    }
  }
  return 0;
}

int attn_fwd(const AttnArgs& a, bf16* Y, float* lse, int B, int N, void* scratch, cudaStream_t stream) {
  if (a.wqk == 128 && a.wv == 128) return launch_flash_fwd<128, 128>(a, Y, lse, B, N, stream);
  if (a.wqk == 128 && a.wv == 64) return launch_flash_fwd<128, 64>(a, Y, lse, B, N, stream);
  if (a.wqk == 64 && a.wv == 64) return launch_flash_fwd<64, 64>(a, Y, lse, B, N, stream);
  return attn_fwd_materialized(a, Y, lse, B, N, scratch, stream);   // other widths: exact chunked path
}

int flash_fwd(const bf16* P3, bf16* Y, float* lse, int B, int N, int Ci, void* scratch, cudaStream_t stream) {
  return attn_fwd(attn_args_embedded(P3, nullptr, Ci), Y, lse, B, N, scratch, stream);
}

static int attn_bwd_materialized(const AttnArgs& a, const bf16* Y, const bf16* dY, const float* lse, float* delta,
                                 float* cs_t, float* cs_p, float* cs_g, ColTables* cs, int B, int N,
                                 void* scratch, cudaStream_t stream) {
  const int ld = attn_ld(N);
  const int nb = attn_chunk(B, N);
  const size_t per = static_cast<size_t>(ld) * N;
  float* S = reinterpret_cast<float*>(scratch);
  float* dPm = S + nb * per;
  bf16* Pm = reinterpret_cast<bf16*>(dPm + nb * per);
  bf16* dS = Pm + nb * per;
  const long long n = N;
  const long long rows = static_cast<long long>(B) * N;
  // bias sums: over all three outputs (mode='embedded': theta / phi / g biases), or over dV alone (mode='gaussian':
  // Q = K = X carry no bias)
  if (!a.bias_qkv) cs_t = cs_p = nullptr;
  // rows of each column-stat table written so far: the three products can leave different row counts per chunk (the
  // dQ GEMM runs 256-row super-tiles for N >= 1024, the other two do not), so each table has its own offset
  int cs_rows_total[3] = {0, 0, 0};
  {
    const long long threads = rows * 32;
    rowdot_kernel<<<static_cast<unsigned>((threads + 255) / 256), 256, 0, stream>>>(dY, Y, delta, rows, a.wv);
    int rc = check_cuda(cudaGetLastError(), "rowdot launch");
    if (rc) return rc;
  }
  for (int b0 = 0; b0 < B; b0 += nb) {
    const int cb = (B - b0 < nb) ? (B - b0) : nb;
    const bf16* Qb = a.q + b0 * n * a.ldq;
    const bf16* Kb = a.k + b0 * n * a.ldk;
    const bf16* Vb = a.v + b0 * n * a.ldv;
    const bf16* dYb = dY + b0 * n * a.wv;
    int r_t = 0, r_p = 0, r_g = 0;
    int rc;
    {  // S = Q K^T (recompute)
      GemmArgs g;
      g.A = opnd(Qb, 0, a.ldq, n * a.ldq);
      g.B = opnd(Kb, 0, a.ldk, n * a.ldk);
      g.B.rows = N;
      g.M = N; g.N = ld; g.K = a.wqk; g.batch = cb;
      g.out_kind = 1;
      g.D = S; g.ldd = ld; g.strideD = static_cast<long long>(per);
      if ((rc = gemm(g, stream))) return rc;
    }
    {  // dPm = dY V^T
      GemmArgs g;
      g.A = opnd(dYb, 0, a.wv, n * a.wv);
      g.B = opnd(Vb, 0, a.ldv, n * a.ldv);
      g.B.rows = N;
      g.M = N; g.N = ld; g.K = a.wv; g.batch = cb;
      g.out_kind = 1;
      g.D = dPm; g.ldd = ld; g.strideD = static_cast<long long>(per);
      if ((rc = gemm(g, stream))) return rc;
    }
    {
      dim3 grid((ld + 255) / 256 > 8 ? 8 : (ld + 255) / 256, static_cast<unsigned>(cb) * N);
      if (grid.y > 65535) {
        // split rows over several launches
        const long long total = static_cast<long long>(cb) * N;
        for (long long r0 = 0; r0 < total; r0 += 65535) {
          dim3 g2(grid.x, static_cast<unsigned>(total - r0 < 65535 ? total - r0 : 65535));
          softmax_bwd_kernel<<<g2, 256, 0, stream>>>(S + r0 * ld, dPm + r0 * ld, lse + static_cast<long long>(b0) * N + r0,
                                                     delta + static_cast<long long>(b0) * N + r0, Pm + r0 * ld,
                                                     dS + r0 * ld, N, ld);
        }
      } else {
        softmax_bwd_kernel<<<grid, 256, 0, stream>>>(S, dPm, lse + static_cast<long long>(b0) * N,
                                                     delta + static_cast<long long>(b0) * N, Pm, dS, N, ld);
      }
      if ((rc = check_cuda(cudaGetLastError(), "softmax_bwd launch"))) return rc;
    }
    {  // dQ = dS K
      GemmArgs g;
      g.A = opnd(dS, 0, ld, static_cast<long long>(per));
      g.B = opnd(Kb, 1, a.ldk, n * a.ldk);
      g.M = N; g.N = a.wqk; g.K = N; g.batch = cb;
      g.D = a.dq + b0 * n * a.ld_dq; g.ldd = a.ld_dq; g.strideD = n * a.ld_dq;
      if (cs_t != nullptr) {
        g.colstats = cs_t + static_cast<long long>(cs_rows_total[0]) * 2 * a.wqk;
        g.colstats_rows = &r_t;
      }
      if ((rc = gemm(g, stream))) return rc;
    }
    {  // dK = dS^T Q
      GemmArgs g;
      g.A = opnd(dS, 1, ld, static_cast<long long>(per));
      g.B = opnd(Qb, 1, a.ldq, n * a.ldq);
      g.M = N; g.N = a.wqk; g.K = N; g.batch = cb;
      g.D = a.dk + b0 * n * a.ld_dk; g.ldd = a.ld_dk; g.strideD = n * a.ld_dk;
      if (cs_p != nullptr) {
        g.colstats = cs_p + static_cast<long long>(cs_rows_total[1]) * 2 * a.wqk;
        g.colstats_rows = &r_p;
      }
      if ((rc = gemm(g, stream))) return rc;
    }
    {  // dV = P^T dY
      GemmArgs g;
      g.A = opnd(Pm, 1, ld, static_cast<long long>(per));
      g.B = opnd(dYb, 1, a.wv, n * a.wv);
      g.M = N; g.N = a.wv; g.K = N; g.batch = cb;
      g.D = a.dvo + b0 * n * a.ld_dv; g.ldd = a.ld_dv; g.strideD = n * a.ld_dv;
      g.colstats = cs_g + static_cast<long long>(cs_rows_total[2]) * 2 * a.wv;
      g.colstats_rows = &r_g;
      if ((rc = gemm(g, stream))) return rc;
    }
    cs_rows_total[0] += r_t;
    cs_rows_total[1] += r_p;
    cs_rows_total[2] += r_g;
  }
  // (embedded: wqk = wv, so the three tables share the row stride 2 wv)
  if (a.bias_qkv) {
    cs->n = 3;
    cs->tab[0] = cs_t; cs->tab[1] = cs_p; cs->tab[2] = cs_g;
    for (int i = 0; i < 3; ++i) cs->rows[i] = cs_rows_total[i];
  } else {
    cs->n = 1;
    cs->tab[0] = cs_g;
    cs->rows[0] = cs_rows_total[2];
  }
  cs->stride = 2LL * a.wv;
  return 0;
}

int flash_bwd_colsum_blocks(long long rows) {
  long long b = (rows + 3) / 4;
  return static_cast<int>(b < 1 ? 1 : (b > 148 * 4 ? 148 * 4 : b));
}

int attn_bwd(const AttnArgs& a, const bf16* Y, const bf16* dY, const float* lse, float* delta, float* cs_t, float* cs_p,
             float* cs_g, int cs_cap_rows, ColTables* cs, int B, int N, void* scratch, cudaStream_t stream) {
  if (!attn_flash_supported(a.wqk, a.wv))   // other widths: exact chunked path
    return attn_bwd_materialized(a, Y, dY, lse, delta, cs_t, cs_p, cs_g, cs, B, N, scratch, stream);
  const long long rows = static_cast<long long>(B) * N;
  {
    const long long threads = rows * 32;
    rowdot_kernel<<<static_cast<unsigned>((threads + 255) / 256), 256, 0, stream>>>(dY, Y, delta, rows, a.wv);
    int rc = check_cuda(cudaGetLastError(), "rowdot launch");
    if (rc) return rc;
  }
  int rc = (a.wqk == 128 && a.wv == 128) ? launch_flash_bwd<128, 128>(a, dY, lse, delta, B, N, stream)
           : (a.wqk == 128)              ? launch_flash_bwd<128, 64>(a, dY, lse, delta, B, N, stream)
                                         : launch_flash_bwd<64, 64>(a, dY, lse, delta, B, N, stream);
  if (rc) return rc;
  int grid = flash_bwd_colsum_blocks(rows);
  if (a.bias_qkv) {
    // bias gradients: column sums of dP3 = [dTheta | dPhi | dG] in one pass, a [grid][2][3Ci] table in cs_t whose
    // column slices are the three tables (cs_p / cs_g are unused here)
    if (grid > cs_cap_rows / 3) grid = cs_cap_rows / 3 > 0 ? cs_cap_rows / 3 : 1;   // cs_t holds cs_cap_rows x 2 x Ci floats
    colsum_bf16_kernel<<<grid, 256, 0, stream>>>(a.dq, cs_t, rows, 3 * a.wv, 3LL * a.wv);
    if ((rc = check_cuda(cudaGetLastError(), "colsum launch"))) return rc;
    cs->n = 3;
    for (int i = 0; i < 3; ++i) {
      cs->tab[i] = cs_t + i * a.wv;
      cs->rows[i] = grid;
    }
    cs->stride = 2LL * 3 * a.wv;
    return 0;
  }
  // column sums of dV alone: a table [grid][2][DV] in cs_g
  if (grid > cs_cap_rows) grid = cs_cap_rows > 0 ? cs_cap_rows : 1;
  colsum_bf16_kernel<<<grid, 256, 0, stream>>>(a.dvo, cs_g, rows, a.wv, a.ld_dv);
  if ((rc = check_cuda(cudaGetLastError(), "colsum launch"))) return rc;
  cs->n = 1;
  cs->tab[0] = cs_g;
  cs->rows[0] = grid;
  cs->stride = 2LL * a.wv;
  return 0;
}

int flash_bwd(const bf16* P3, const bf16* Y, const bf16* dY, const float* lse, bf16* dP3, float* delta, float* cs_t,
              float* cs_p, float* cs_g, int cs_cap_rows, ColTables* cs, int B, int N, int Ci, void* scratch,
              cudaStream_t stream) {
  return attn_bwd(attn_args_embedded(P3, dP3, Ci), Y, dY, lse, delta, cs_t, cs_p, cs_g, cs_cap_rows, cs, B, N, scratch,
                  stream);
}

// out[r, c] = in[r, c] + in[r, C + c] over rows of 2C bf16 (fp32 sum, one rounding): dS X + dS^T X of mode='gaussian'
__global__ void __launch_bounds__(256) sum_halves_kernel(const bf16* __restrict__ in, bf16* __restrict__ out,
                                                        long long rows, int C) {
  const long long nvec = rows * (C / 8);
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < nvec;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / (C / 8);
    const int c = static_cast<int>(i % (C / 8)) * 8;
    const uint4 a = *reinterpret_cast<const uint4*>(in + r * 2 * C + c);
    const uint4 b = *reinterpret_cast<const uint4*>(in + r * 2 * C + C + c);
    const uint32_t* ua = reinterpret_cast<const uint32_t*>(&a);
    const uint32_t* ub = reinterpret_cast<const uint32_t*>(&b);
    uint4 o;
    uint32_t* uo = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const float2 x = unpack_bf16(ua[t]), y = unpack_bf16(ub[t]);
      uo[t] = pack_bf16(x.x + y.x, x.y + y.y);
    }
    *reinterpret_cast<uint4*>(out + r * C + c) = o;
  }
}

int sum_halves(const bf16* in, bf16* out, long long rows, int C, cudaStream_t stream) {
  const long long nvec = rows * (C / 8);
  long long blocks = (nvec + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks < 1) blocks = 1;
  sum_halves_kernel<<<static_cast<unsigned>(blocks), 256, 0, stream>>>(in, out, rows, C);
  return check_cuda(cudaGetLastError(), "sum_halves launch");
}

}  // namespace glf
