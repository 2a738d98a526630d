// glf_ln.cu — bulk-copy (TMA engine) staged versions of the two HBM-bound row kernels of the fusion path,
//   forward : Z = sum_m LayerNorm_C(a_m * U_m + b_m + X_m) * lw_m + lb_m        (ours.py:908-915; m = MGFM, MLFM)
//   backward: dV_m = d(pre-LayerNorm sum) and per-CTA partials of the four per-channel reductions
// for bf16 activations with C <= 256 (one warp owns a row, one lane 8 channels).  Z / dZ, the tensors the caller hands
// over or receives, are bf16 or fp16 (TZ): the same bytes per row, converted where they are read or written.
//
// Why: the register-prefetch kernels of glf_eltwise.cu keep ~24 KB per SM in flight, B200 needs roughly twice that to
// saturate HBM3e (measured 60-75 % of the copy bandwidth).  Here one producer warp streams contiguous row tiles
// (rows are contiguous in token-major activations, so a tile is ONE cp.async.bulk per tensor, no tensor map) into a
// shared-memory ring — 180-215 KB in flight per SM — and 14-15 consumer warps read rows from shared memory.
// NMOD = 2 is the "pair" form used by the fused MGFM + MLFM call site: both blocks' LayerNorms in one pass, so dZ
// (backward) and Z (forward, the `global + local` sum of ours.py:1834) cross HBM once instead of twice.
// Determinism: per-CTA partials, fixed-order combination — same contract as the register kernels.
#include "glf_internal.h"
#include "glf_ptx.cuh"

namespace glf {

namespace {

__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

// 8 16-bit elements (bf16 or fp16) from shared memory as four float2 (element pairs)
template <typename T = bf16>
__device__ __forceinline__ void lds8p(const uint8_t* p, float2 (&f)[4]) {
  const uint4 v = *reinterpret_cast<const uint4*>(p);
  const uint32_t* u = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) f[i] = unpack2<T>(u[i]);
}
__device__ __forceinline__ void ldg8p(const float* p, float2 (&f)[4]) {
  const float4 a = *reinterpret_cast<const float4*>(p);
  const float4 b = *reinterpret_cast<const float4*>(p + 4);
  f[0] = make_float2(a.x, a.y); f[1] = make_float2(a.z, a.w);
  f[2] = make_float2(b.x, b.y); f[3] = make_float2(b.z, b.w);
}
template <typename T>
__device__ __forceinline__ void stg8p(T* p, const float2 (&f)[4]) {
  *reinterpret_cast<uint4*>(p) = make_uint4(pack2<T>(f[0].x, f[0].y), pack2<T>(f[1].x, f[1].y),
                                            pack2<T>(f[2].x, f[2].y), pack2<T>(f[3].x, f[3].y));
}
__device__ __forceinline__ float hsum4(const float2 (&f)[4]) {
  const float2 t = add2(add2(f[0], f[1]), add2(f[2], f[3]));
  return t.x + t.y;
}
__device__ __forceinline__ float2 splat(float x) { return make_float2(x, x); }


constexpr int MAX_STAGES = 8;
constexpr uint32_t RING_BUDGET = 218 * 1024;

// ------------------------------------------------------------------------------------------------ forward
constexpr int F_CW = 15;               // consumer warps
constexpr int F_TR = 2 * F_CW;         // rows per tile (two per consumer warp)
constexpr int F_THREADS = (F_CW + 1) * 32;

struct LnFwdParams {
  const bf16* U[2];
  const bf16* X[2];
  const float* a[2];
  const float* b[2];
  const float* lw[2];
  const float* lb[2];
  float* mu[2];
  float* r[2];
  void* Z;         // [rows, C] of the kernel's TZ
  void* Z0;        // PARTS only: the first module's own output (MGFM's f4_global_fusion, ours.py:1823), TZ [rows, C]
  long long rows;
  int C, ntiles, stages, accumulate;
  uint32_t arr_bytes, stage_bytes;
  float eps;
};

// FULLC: C == 256, every lane owns 8 live channels.  PARTS: also store module 0's LayerNorm output on its own (the
// cycle-consistency pass of the trainer, R/main.py:211-235, consumes f4_global_fusion beside the fused sum).
template <int NMOD, bool FULLC, bool PARTS, typename TZ>
__global__ void __launch_bounds__(F_THREADS, 1) ln_fwd_tma_kernel(const LnFwdParams p) {
  extern __shared__ uint8_t lsm_raw[];
  __shared__ uint64_t full_bar[MAX_STAGES], empty_bar[MAX_STAGES];
  const uint32_t pad = (128u - (smem_u32(lsm_raw) & 127u)) & 127u;
  uint8_t* ring = lsm_raw + pad;
  const uint32_t ring_u32 = smem_u32(ring);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int narr = 2 * NMOD + (p.accumulate ? 1 : 0);
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), F_CW);
    }
    fence_mbar_init();
  }
  __syncthreads();

  if (warp == F_CW) {
    // ------------------------------------------------------------------------------------------ producer
    if (elect_one()) {
      int it = 0;
      for (int t = blockIdx.x; t < p.ntiles; t += gridDim.x, ++it) {
        const int s = it % p.stages;
        const uint32_t ph = static_cast<uint32_t>(it / p.stages) & 1u;
        mbar_wait(smem_u32(&empty_bar[s]), ph ^ 1u);
        const long long row0 = static_cast<long long>(t) * F_TR;
        const long long left = p.rows - row0;
        const uint32_t nrow = static_cast<uint32_t>(left < F_TR ? left : F_TR);
        const uint32_t bytes = nrow * static_cast<uint32_t>(p.C) * 2u;
        const uint32_t fb = smem_u32(&full_bar[s]);
        mbar_expect_tx(fb, bytes * narr);
        const uint32_t dst = ring_u32 + s * p.stage_bytes;
        const long long off = row0 * p.C;
#pragma unroll
        for (int m = 0; m < NMOD; ++m) {
          bulk_g2s(dst + (2 * m) * p.arr_bytes, p.U[m] + off, bytes, fb);
          bulk_g2s(dst + (2 * m + 1) * p.arr_bytes, p.X[m] + off, bytes, fb);
        }
        if (p.accumulate) bulk_g2s(dst + 2 * NMOD * p.arr_bytes, reinterpret_cast<const TZ*>(p.Z) + off, bytes, fb);
      }
    }
    return;
  }
  // -------------------------------------------------------------------------------------------- consumers
  // all per-element math on float2 pairs (FFMA2 / FADD2 / FMUL2): the kernel is instruction-issue bound otherwise
  const int c0 = lane * 8;
  const bool cact = FULLC || c0 < p.C;
  float2 pa[NMOD][4], pb[NMOD][4], pw[NMOD][4], plsum[4], plb0[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) plsum[i] = plb0[i] = splat(0.f);
#pragma unroll
  for (int m = 0; m < NMOD; ++m) {
#pragma unroll
    for (int i = 0; i < 4; ++i) pa[m][i] = pb[m][i] = pw[m][i] = splat(0.f);
    if (cact) {
      float2 lb[4];
      ldg8p(p.a[m] + c0, pa[m]);
      ldg8p(p.b[m] + c0, pb[m]);
      ldg8p(p.lw[m] + c0, pw[m]);
      ldg8p(p.lb[m] + c0, lb);
#pragma unroll
      for (int i = 0; i < 4; ++i) plsum[i] = add2(plsum[i], lb[i]);
      if (PARTS && m == 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) plb0[i] = lb[i];
      }
    }
  }
  const float invC = 1.f / static_cast<float>(p.C);
  const uint32_t row_bytes = static_cast<uint32_t>(p.C) * 2u;
  int it = 0;
  for (int t = blockIdx.x; t < p.ntiles; t += gridDim.x, ++it) {
    const int s = it % p.stages;
    const uint32_t ph = static_cast<uint32_t>(it / p.stages) & 1u;
    const long long row0 = static_cast<long long>(t) * F_TR;
    const long long left = p.rows - row0;
    const int nrow = static_cast<int>(left < F_TR ? left : F_TR);
    mbar_wait(smem_u32(&full_bar[s]), ph);
    const uint8_t* st = ring + s * p.stage_bytes;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int rl = warp + k * F_CW;
      if (rl < nrow) {
        const long long row = row0 + rl;
        const uint32_t roff = rl * row_bytes + c0 * 2;
        float2 o[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) o[i] = plsum[i];
        if (cact && p.accumulate) {
          float2 z0[4];
          lds8p<TZ>(st + 2 * NMOD * p.arr_bytes + roff, z0);
#pragma unroll
          for (int i = 0; i < 4; ++i) o[i] = add2(o[i], z0[i]);
        }
        // both blocks' rows go through the two warp reductions TOGETHER (same two-pass arithmetic per block, half the
        // dependent shuffle chains per row)
        float2 v[NMOD][4];
        float red[NMOD];
#pragma unroll
        for (int m = 0; m < NMOD; ++m) {
#pragma unroll
          for (int i = 0; i < 4; ++i) v[m][i] = splat(0.f);
          if (cact) {
            float2 u[4], x[4];
            lds8p(st + (2 * m) * p.arr_bytes + roff, u);
            lds8p(st + (2 * m + 1) * p.arr_bytes + roff, x);
#pragma unroll
            for (int i = 0; i < 4; ++i) v[m][i] = add2(fma2(pa[m][i], u[i], pb[m][i]), x[i]);
          }
          red[m] = hsum4(v[m]);
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
#pragma unroll
          for (int m = 0; m < NMOD; ++m) red[m] += __shfl_xor_sync(0xffffffffu, red[m], off);
        }
        float mu[NMOD];
#pragma unroll
        for (int m = 0; m < NMOD; ++m) {
          mu[m] = red[m] * invC;
          const float2 nmu = splat(-mu[m]);
          float2 q2 = splat(0.f);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            v[m][i] = cact ? add2(v[m][i], nmu) : splat(0.f);     // v now holds the centred values
            q2 = fma2(v[m][i], v[m][i], q2);
          }
          red[m] = q2.x + q2.y;
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
#pragma unroll
          for (int m = 0; m < NMOD; ++m) red[m] += __shfl_xor_sync(0xffffffffu, red[m], off);
        }
#pragma unroll
        for (int m = 0; m < NMOD; ++m) {
          const float r = rsqrtf(red[m] * invC + p.eps);
          const float2 r2 = splat(r);
#pragma unroll
          for (int i = 0; i < 4; ++i) o[i] = fma2(v[m][i], mul2(pw[m][i], r2), o[i]);
          if (PARTS && m == 0 && cact) {
            float2 o0[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) o0[i] = fma2(v[0][i], mul2(pw[0][i], r2), plb0[i]);
            stg8p(reinterpret_cast<TZ*>(p.Z0) + row * p.C + c0, o0);
          }
          if (lane == 0 && p.mu[m] != nullptr) {
            p.mu[m][row] = mu[m];
            p.r[m][row] = r;
          }
        }
        if (cact) stg8p(reinterpret_cast<TZ*>(p.Z) + row * p.C + c0, o);
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(smem_u32(&empty_bar[s]));
  }
}

// ------------------------------------------------------------------------------------------------ backward
constexpr int B_CW = 14;               // consumer warps (two groups of 7 in the pair form)
constexpr int B_TR = 28;               // rows per tile
constexpr int B_THREADS = (B_CW + 1) * 32;
constexpr int B_ACC_PITCH = 256 + 8;

struct LnBwdParams {
  const void* dZ;            // [rows, C] of the kernel's TZ
  const bf16* U[2];
  const bf16* X[2];
  const float* a[2];
  const float* b[2];
  const float* lw[2];
  const float* bn_mean[2];
  const float* bn_rstd[2];
  const float* mu[2];
  const float* r[2];
  bf16* dV[2];
  float* part[2];
  long long rows;
  int C, ntiles, stages;
  uint32_t arr_bytes, stage_bytes;
  // dZ given per view (the dict-keyed call site: one gradient per view, rows of C channels): row (b, v, t) of the stack
  // lives at dzv[v] + b * dz_sb[v] + t * C.  dz_nv = 0: dZ is the token-major stack itself.  Needs hw % B_TR == 0 so
  // that a tile never straddles two views.
  const void* dzv[8];
  long long dz_sb[8];
  int dz_nv, dz_hw;
};

template <int NMOD, bool FULLC, typename TZ>
__global__ void __launch_bounds__(B_THREADS, 1) ln_bwd_tma_kernel(const LnBwdParams p) {
  extern __shared__ uint8_t lsm_raw[];
  __shared__ uint64_t full_bar[MAX_STAGES], empty_bar[MAX_STAGES];
  const uint32_t pad = (128u - (smem_u32(lsm_raw) & 127u)) & 127u;
  uint8_t* ring = lsm_raw + pad;
  const uint32_t ring_u32 = smem_u32(ring);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // stage layout: dZ | (U_m | X_m) x NMOD | (mu_m | r_m) x NMOD   (the per-row statistics are 128-byte slots)
  const uint32_t stat_off = (1 + 2 * NMOD) * p.arr_bytes;
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), B_CW);
    }
    fence_mbar_init();
  }
  __syncthreads();

  if (warp == B_CW) {
    if (elect_one()) {
      int it = 0;
      for (int t = blockIdx.x; t < p.ntiles; t += gridDim.x, ++it) {
        const int s = it % p.stages;
        const uint32_t ph = static_cast<uint32_t>(it / p.stages) & 1u;
        mbar_wait(smem_u32(&empty_bar[s]), ph ^ 1u);
        const long long row0 = static_cast<long long>(t) * B_TR;
        const long long left = p.rows - row0;
        const uint32_t nrow = static_cast<uint32_t>(left < B_TR ? left : B_TR);
        const uint32_t bytes = nrow * static_cast<uint32_t>(p.C) * 2u;
        const bool full_tile = nrow == B_TR;     // per-row statistics ride along only for full tiles (16-byte sizes)
        const uint32_t fb = smem_u32(&full_bar[s]);
        mbar_expect_tx(fb, bytes * (1 + 2 * NMOD) + (full_tile ? 2u * NMOD * B_TR * 4u : 0u));
        const uint32_t dst = ring_u32 + s * p.stage_bytes;
        const long long off = row0 * p.C;
        const TZ* dzsrc = reinterpret_cast<const TZ*>(p.dZ) + off;
        if (p.dz_nv > 0) {
          const long long bv = row0 / p.dz_hw;
          const int v = static_cast<int>(bv % p.dz_nv);
          dzsrc = reinterpret_cast<const TZ*>(p.dzv[v]) + (bv / p.dz_nv) * p.dz_sb[v] + (row0 - bv * p.dz_hw) * p.C;
        }
        bulk_g2s(dst, dzsrc, bytes, fb);
#pragma unroll
        for (int m = 0; m < NMOD; ++m) {
          bulk_g2s(dst + (1 + 2 * m) * p.arr_bytes, p.U[m] + off, bytes, fb);
          bulk_g2s(dst + (2 + 2 * m) * p.arr_bytes, p.X[m] + off, bytes, fb);
          if (full_tile) {
            bulk_g2s(dst + stat_off + (2 * m) * 128, p.mu[m] + row0, B_TR * 4, fb);
            bulk_g2s(dst + stat_off + (2 * m + 1) * 128, p.r[m] + row0, B_TR * 4, fb);
          }
        }
      }
    }
  } else {
    constexpr int GW = B_CW / NMOD;              // warps per module group
    constexpr int RPW = B_TR / GW;               // rows per warp per tile
    const int m = (NMOD == 2) ? warp / GW : 0;   // module of this warp
    const int wi = warp % GW;
    const int c0 = lane * 8;
    const bool cact = FULLC || c0 < p.C;
    float2 pa[4], pb[4], pw[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) pa[i] = pb[i] = pw[i] = splat(0.f);
    if (cact) {
      ldg8p(p.a[m] + c0, pa);
      ldg8p(p.b[m] + c0, pb);
      ldg8p(p.lw[m] + c0, pw);
    }
    float2 g_lw[4], g_lb[4], g_ga[4], g_be[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) g_lw[i] = g_lb[i] = g_ga[i] = g_be[i] = splat(0.f);
    const float invC = 1.f / static_cast<float>(p.C);
    const uint32_t row_bytes = static_cast<uint32_t>(p.C) * 2u;
    const uint32_t u_off = (1 + 2 * m) * p.arr_bytes, x_off = (2 + 2 * m) * p.arr_bytes;
    bf16* dVm = p.dV[m];
    int it = 0;
    for (int t = blockIdx.x; t < p.ntiles; t += gridDim.x, ++it) {
      const int s = it % p.stages;
      const uint32_t ph = static_cast<uint32_t>(it / p.stages) & 1u;
      const long long row0 = static_cast<long long>(t) * B_TR;
      const long long left = p.rows - row0;
      const int nrow = static_cast<int>(left < B_TR ? left : B_TR);
      const bool full_tile = nrow == B_TR;
      mbar_wait(smem_u32(&full_bar[s]), ph);
      const uint8_t* st = ring + s * p.stage_bytes;
      const float* mu_s = reinterpret_cast<const float*>(st + stat_off + (2 * m) * 128);
      const float* r_s = reinterpret_cast<const float*>(st + stat_off + (2 * m + 1) * 128);
#pragma unroll
      for (int k = 0; k < RPW; ++k) {
        const int rl = wi + k * GW;
        if (rl < nrow) {
          const long long row = row0 + rl;
          const float mu = full_tile ? mu_s[rl] : p.mu[m][row];
          const float r = full_tile ? r_s[rl] : p.r[m][row];
          const uint32_t roff = rl * row_bytes + c0 * 2;
          float2 xh[4], dxh[4], dz[4], u[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) xh[i] = dxh[i] = dz[i] = u[i] = splat(0.f);
          if (cact) {
            float2 x[4];
            lds8p<TZ>(st + roff, dz);
            lds8p(st + u_off + roff, u);
            lds8p(st + x_off + roff, x);
            const float2 r2 = splat(r), nmur = splat(-mu * r);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              // xhat = (a u + b + x - mu) r = (a u + b + x) r - mu r
              xh[i] = fma2(add2(fma2(pa[i], u[i], pb[i]), x[i]), r2, nmur);
              dxh[i] = mul2(dz[i], pw[i]);
            }
          }
          float2 s1p = splat(0.f);
#pragma unroll
          for (int i = 0; i < 4; ++i) s1p = fma2(dxh[i], xh[i], s1p);
          const float s0 = warp_sum(hsum4(dxh));
          const float s1 = warp_sum(s1p.x + s1p.y);
          if (cact) {
            const float2 nm1 = splat(-s0 * invC), nm2 = splat(-s1 * invC), r2 = splat(r);
            float2 dv[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              dv[i] = mul2(r2, fma2(xh[i], nm2, add2(dxh[i], nm1)));
              g_lw[i] = fma2(dz[i], xh[i], g_lw[i]);
              g_lb[i] = add2(g_lb[i], dz[i]);
              g_ga[i] = fma2(dv[i], u[i], g_ga[i]);    // raw U: turned into sum dv * uhat when the partial is written
              g_be[i] = add2(g_be[i], dv[i]);
            }
            stg8p(dVm + row * p.C + c0, dv);
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&empty_bar[s]));
    }
    // every tile has been consumed (so every bulk copy has landed): the ring storage is free for the exchange
    named_bar_sync(1, B_CW * 32);
    float(*acc)[4][B_ACC_PITCH] = reinterpret_cast<float(*)[4][B_ACC_PITCH]>(ring);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      *reinterpret_cast<float2*>(&acc[warp][0][c0 + 2 * i]) = g_lw[i];
      *reinterpret_cast<float2*>(&acc[warp][1][c0 + 2 * i]) = g_lb[i];
      *reinterpret_cast<float2*>(&acc[warp][2][c0 + 2 * i]) = g_ga[i];
      *reinterpret_cast<float2*>(&acc[warp][3][c0 + 2 * i]) = g_be[i];
    }
    named_bar_sync(1, B_CW * 32);
    // one partial row per CTA and module: [4][C]; index space = NMOD x C channels
    for (int idx = threadIdx.x; idx < NMOD * p.C; idx += B_CW * 32) {
      const int mm = idx / p.C, c = idx % p.C;
      float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
      for (int w = mm * GW; w < (mm + 1) * GW; ++w) {
        t0 += acc[w][0][c];
        t1 += acc[w][1][c];
        t2 += acc[w][2][c];
        t3 += acc[w][3][c];
      }
      // sum dv * uhat = rstd * (sum dv * u - mean * sum dv)
      const float ga = p.bn_rstd[mm][c] * (t2 - p.bn_mean[mm][c] * t3);
      float* out = p.part[mm] + static_cast<long long>(blockIdx.x) * 4 * p.C;
      out[c] = t0;
      out[p.C + c] = t1;
      out[2 * p.C + c] = ga;
      out[3 * p.C + c] = t3;
    }
  }
}

int num_sms() {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
    return 148;
  return n > 0 ? n : 148;
}

}  // namespace

bool ln_tma_supported(int C) { return C % 8 == 0 && C <= 256 && C >= 8; }

int ln_bwd_tma_blocks(long long rows) {
  const long long nt = (rows + B_TR - 1) / B_TR;
  const int sms = 148;   // partial-table capacity is sized for 2 * 148 rows (glf_bn_res_ln_bwd_max_blocks)
  return static_cast<int>(nt < sms ? nt : sms);
}

// Z (+)= sum over the nmod modules of LayerNorm(a U + b + X) lw + lb.  U, X bf16 [rows, C]; Z (and Z0) of z_dtype.
int ln_fwd_tma(int nmod, const bf16* const* U, const bf16* const* X, const float* const* a, const float* const* b,
               const float* const* lw, const float* const* lb, float* const* mu, float* const* r, void* Z,
               long long rows, int C, float eps, int accumulate, cudaStream_t stream, void* Z0, int z_dtype) {
  if (!ln_tma_supported(C) || nmod < 1 || nmod > 2) return set_error(GLF_ERR_INVALID, "ln_fwd_tma: unsupported shape");
  if (z_dtype != GLF_DTYPE_BF16 && z_dtype != GLF_DTYPE_F16) return set_error(GLF_ERR_INVALID, "ln_fwd_tma: Z must be bf16 or fp16");
  if (Z0 != nullptr && nmod != 2) return set_error(GLF_ERR_INVALID, "ln_fwd_tma: the parts output needs both modules");
  LnFwdParams p;
  p.Z0 = Z0;
  for (int m = 0; m < 2; ++m) {
    const int k = m < nmod ? m : 0;
    p.U[m] = U[k]; p.X[m] = X[k]; p.a[m] = a[k]; p.b[m] = b[k]; p.lw[m] = lw[k]; p.lb[m] = lb[k];
    p.mu[m] = mu ? mu[k] : nullptr;
    p.r[m] = r ? r[k] : nullptr;
  }
  p.Z = Z; p.rows = rows; p.C = C; p.eps = eps; p.accumulate = accumulate ? 1 : 0;
  p.ntiles = static_cast<int>((rows + F_TR - 1) / F_TR);
  p.arr_bytes = static_cast<uint32_t>(F_TR) * C * 2;
  p.arr_bytes = (p.arr_bytes + 127u) & ~127u;
  p.stage_bytes = p.arr_bytes * (2 * nmod + (accumulate ? 1 : 0));
  int stages = static_cast<int>(RING_BUDGET / p.stage_bytes);
  p.stages = stages > MAX_STAGES ? MAX_STAGES : (stages < 2 ? 2 : stages);
  const uint32_t smem = p.stages * p.stage_bytes + 128;
  const int sms = num_sms();
  const int grid = p.ntiles < sms ? p.ntiles : sms;
  const bool h = z_dtype == GLF_DTYPE_F16;
  void (*kern)(const LnFwdParams);
  if (Z0 != nullptr)
    kern = C == 256 ? (h ? ln_fwd_tma_kernel<2, true, true, f16> : ln_fwd_tma_kernel<2, true, true, bf16>)
                    : (h ? ln_fwd_tma_kernel<2, false, true, f16> : ln_fwd_tma_kernel<2, false, true, bf16>);
  else if (nmod == 2)
    kern = C == 256 ? (h ? ln_fwd_tma_kernel<2, true, false, f16> : ln_fwd_tma_kernel<2, true, false, bf16>)
                    : (h ? ln_fwd_tma_kernel<2, false, false, f16> : ln_fwd_tma_kernel<2, false, false, bf16>);
  else
    kern = C == 256 ? (h ? ln_fwd_tma_kernel<1, true, false, f16> : ln_fwd_tma_kernel<1, true, false, bf16>)
                    : (h ? ln_fwd_tma_kernel<1, false, false, f16> : ln_fwd_tma_kernel<1, false, false, bf16>);
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(ln_fwd_tma)");
  kern<<<grid, F_THREADS, smem, stream>>>(p);
  return check_cuda(cudaGetLastError(), "ln_fwd_tma launch");
}

int ln_bwd_tma_tile_rows() { return B_TR; }

// dV_m and per-CTA partials [blocks][4][C] per module; returns the number of partial rows through *nblocks.  dZ (or the
// per-view dz) of dz_dtype.
int ln_bwd_tma(int nmod, const void* dZ, const bf16* const* U, const bf16* const* X, const float* const* a,
               const float* const* b, const float* const* lw, const float* const* bn_mean,
               const float* const* bn_rstd, const float* const* mu, const float* const* r, bf16* const* dV,
               float* const* part, long long rows, int C, int* nblocks, cudaStream_t stream, int dz_nv,
               const void* const* dz_views, const long long* dz_sb, int dz_hw, int dz_dtype) {
  if (!ln_tma_supported(C) || nmod < 1 || nmod > 2) return set_error(GLF_ERR_INVALID, "ln_bwd_tma: unsupported shape");
  if (dz_dtype != GLF_DTYPE_BF16 && dz_dtype != GLF_DTYPE_F16) return set_error(GLF_ERR_INVALID, "ln_bwd_tma: dZ must be bf16 or fp16");
  LnBwdParams p;
  p.dZ = dZ;
  p.dz_nv = 0; p.dz_hw = 1;
  for (int v = 0; v < 8; ++v) { p.dzv[v] = nullptr; p.dz_sb[v] = 0; }
  if (dz_nv > 0) {
    if (dz_nv > 8 || dz_views == nullptr || dz_sb == nullptr || dz_hw <= 0 || dz_hw % B_TR != 0 ||
        rows % (static_cast<long long>(dz_nv) * dz_hw) != 0)
      return set_error(GLF_ERR_UNSUPPORTED, "ln_bwd_tma: per-view dz needs h*w %% %d == 0 and <= 8 views", B_TR);
    for (int v = 0; v < dz_nv; ++v) {
      if (dz_views[v] == nullptr || (reinterpret_cast<uintptr_t>(dz_views[v]) & 15) != 0 || dz_sb[v] % 8 != 0)
        return set_error(GLF_ERR_INVALID, "ln_bwd_tma: per-view dz must be 16-byte aligned");
      p.dzv[v] = dz_views[v];
      p.dz_sb[v] = dz_sb[v];
    }
    p.dz_nv = dz_nv; p.dz_hw = dz_hw;
    p.dZ = p.dzv[0];
  }
  for (int m = 0; m < 2; ++m) {
    const int k = m < nmod ? m : 0;
    p.U[m] = U[k]; p.X[m] = X[k]; p.a[m] = a[k]; p.b[m] = b[k]; p.lw[m] = lw[k];
    p.bn_mean[m] = bn_mean[k]; p.bn_rstd[m] = bn_rstd[k]; p.mu[m] = mu[k]; p.r[m] = r[k];
    p.dV[m] = dV[k]; p.part[m] = part[k];
  }
  p.rows = rows; p.C = C;
  p.ntiles = static_cast<int>((rows + B_TR - 1) / B_TR);
  p.arr_bytes = static_cast<uint32_t>(B_TR) * C * 2;
  p.arr_bytes = (p.arr_bytes + 127u) & ~127u;
  p.stage_bytes = p.arr_bytes * (1 + 2 * nmod) + 2 * nmod * 128;
  const uint32_t exch = B_CW * 4 * B_ACC_PITCH * sizeof(float);   // accumulator exchange reuses the ring
  int stages = static_cast<int>(RING_BUDGET / p.stage_bytes);
  p.stages = stages > MAX_STAGES ? MAX_STAGES : (stages < 2 ? 2 : stages);
  uint32_t ring_bytes = p.stages * p.stage_bytes;
  if (ring_bytes < exch) ring_bytes = exch;
  const uint32_t smem = ring_bytes + 128;
  const int grid = ln_bwd_tma_blocks(rows);
  if (nblocks) *nblocks = grid;
  const bool h = dz_dtype == GLF_DTYPE_F16;
  void (*kern)(const LnBwdParams) =
      nmod == 2 ? (C == 256 ? (h ? ln_bwd_tma_kernel<2, true, f16> : ln_bwd_tma_kernel<2, true, bf16>)
                            : (h ? ln_bwd_tma_kernel<2, false, f16> : ln_bwd_tma_kernel<2, false, bf16>))
                : (C == 256 ? (h ? ln_bwd_tma_kernel<1, true, f16> : ln_bwd_tma_kernel<1, true, bf16>)
                            : (h ? ln_bwd_tma_kernel<1, false, f16> : ln_bwd_tma_kernel<1, false, bf16>));
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(ln_bwd_tma)");
  kern<<<grid, B_THREADS, smem, stream>>>(p);
  return check_cuda(cudaGetLastError(), "ln_bwd_tma launch");
}

}  // namespace glf
