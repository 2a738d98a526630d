// The cycle-consistency step that consumes the fusion path's MGFM output (R/main.py:229-235):
//   spatial_sums   cyc_feat_out[view].sum(dim=(2, 3))                 R/main.py:229
//   cycle_loss     Trainer.seg_cycle / Trainer.dense_seg_cycle        R/main.py:650-717 / :719-798
// The reference spells the loss with ~60 repeat / gather / softmax launches per start position (and as many again in
// autograd); the gathers are plain shifted reads (their modulo wrap is sliced off again), so one CTA per start
// position evaluates loss_s AND d loss_s / d feat in a single pass, and a second launch adds the positions up in a
// fixed order.  Everything is fp32 SIMT on [T, C] features of a few dozen frames: launch-bound work, not a GEMM.
//
// With K = feat[R:], nk = T - R, a = temperature / (C ch), start s:
//   sim_i = -a sum_j |K[i+j] - feat[s+j]|^2,  beta = softmax(sim),  w_j = sum_i beta_i K[off+i+j],
//   z_m = -a sum_j |feat[off+m+j] - w_j|^2,   loss_s = mean_m BCEWithLogits(z_m, y_m)
#include <cstdint>
#include <type_traits>

#include "glf_internal.h"

namespace glf {

namespace {

constexpr int CY_THREADS = 1024;
constexpr int CY_WARPS = CY_THREADS / 32;
constexpr int CY_MAXPOS = 1024;          // upper bound on the key / query position counts (shared-memory vectors)

struct CycleParams {
  const float* feat;                      // [T, C]
  int T, C, R, off, ch;
  float a;                                // temperature / (C * ch)
  int s0, step, n_starts;
  int soft_label;
  float* part;                            // [n_starts, T, C] per-start gradients
  float* loss_part;                       // [n_starts]
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__global__ void __launch_bounds__(CY_THREADS) cycle_start_kernel(CycleParams P) {
  extern __shared__ float sm[];
  const int C = P.C, ch = P.ch, R = P.R, off = P.off, T = P.T;
  const int nk = T - R, Lk = nk - ch - off + 1, Lq = R - off - ch + 1;
  float* w = sm;                          // [ch][C]
  float* dw = w + ch * C;                 // [ch][C]
  float* beta = dw + ch * C;              // [Lk]   sim, then softmax weights
  float* dsim = beta + Lk;                // [Lk]   d beta, then d sim
  float* dz = dsim + Lk;                  // [Lq]
  __shared__ float red[CY_WARPS];
  __shared__ float bcast;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int s = P.s0 + blockIdx.x * P.step;
  const float a = P.a;
  const float* __restrict__ feat = P.feat;
  const float* __restrict__ K = feat + static_cast<long long>(R) * C;
  const float* __restrict__ q = feat + static_cast<long long>(s) * C;      // q_j = q + j*C
  float* __restrict__ part = P.part + static_cast<long long>(blockIdx.x) * T * C;

  // sim_i (main.py:666-679)
  for (int i = warp; i < Lk; i += CY_WARPS) {
    float acc = 0.f;
    for (int j = 0; j < ch; ++j) {
      const float* kr = K + static_cast<long long>(i + j) * C;
      const float* qr = q + static_cast<long long>(j) * C;
      for (int c = lane; c < C; c += 32) { const float d = kr[c] - qr[c]; acc = fmaf(d, d, acc); }
    }
    acc = warp_sum(acc);
    if (lane == 0) beta[i] = -a * acc;
  }
  __syncthreads();
  // beta = softmax(sim) (main.py:680)
  if (warp == 0) {
    float mx = -INFINITY;
    for (int i = lane; i < Lk; i += 32) mx = fmaxf(mx, beta[i]);
    mx = warp_max(mx);
    float sum = 0.f;
    for (int i = lane; i < Lk; i += 32) { const float e = expf(beta[i] - mx); beta[i] = e; sum += e; }
    sum = warp_sum(sum);
    const float inv = 1.f / sum;
    for (int i = lane; i < Lk; i += 32) beta[i] *= inv;
  }
  __syncthreads();
  // w_j = sum_i beta_i K[off+i+j] (main.py:685-693)
  for (int it = tid; it < ch * C; it += CY_THREADS) {        // one (j, c) pair per thread, coalesced along c
    const int j = it / C, c = it - j * C;
    const float* kc = K + static_cast<long long>(off + j) * C + c;
    float a0 = 0.f, a1 = 0.f;
    int i = 0;
    for (; i + 1 < Lk; i += 2) {
      a0 = fmaf(beta[i], kc[static_cast<long long>(i) * C], a0);
      a1 = fmaf(beta[i + 1], kc[static_cast<long long>(i + 1) * C], a1);
    }
    if (i < Lk) a0 = fmaf(beta[i], kc[static_cast<long long>(i) * C], a0);
    w[it] = a0 + a1;
  }
  __syncthreads();
  // z_m, the loss and d loss / d z (main.py:697-717)
  float bce = 0.f;
  for (int m = warp; m < Lq; m += CY_WARPS) {
    float acc = 0.f;
    for (int j = 0; j < ch; ++j) {
      const float* xr = feat + static_cast<long long>(off + m + j) * C;
      const float* wr = w + j * C;
      for (int c = lane; c < C; c += 32) { const float d = xr[c] - wr[c]; acc = fmaf(d, d, acc); }
    }
    acc = warp_sum(acc);
    if (lane == 0) {
      const float z = -a * acc;
      float y = m == s ? 1.f : 0.f;
      if (P.soft_label) y = m == s ? 0.8f : 0.2f / static_cast<float>(Lq - 1);
      bce += fmaxf(z, 0.f) - z * y + log1pf(expf(-fabsf(z)));
      dz[m] = (1.f / (1.f + expf(-z)) - y) / static_cast<float>(Lq);
    }
  }
  if (lane == 0) red[warp] = bce;
  __syncthreads();
  if (tid == 0) {
    float t = 0.f;
    for (int i = 0; i < CY_WARPS; ++i) t += red[i];
    P.loss_part[blockIdx.x] = t / static_cast<float>(Lq);
  }
  // ---- backward, gather form: every gradient row is written once by the thread that owns its channel, from
  // independent loads (no read-modify-write chains, no atomics; deterministic).
  //   dw_j = 2a sum_m dz_m (feat[off+m+j] - w_j)
  for (int it = tid; it < ch * C; it += CY_THREADS) {
    const int j = it / C, c = it - j * C;
    const float wj = w[it];
    float acc = 0.f;
    for (int m = 0; m < Lq; ++m) acc = fmaf(dz[m], feat[static_cast<long long>(off + m + j) * C + c] - wj, acc);
    dw[it] = 2.f * a * acc;
  }
  __syncthreads();
  // d beta_i = sum_j <dw_j, K[off+i+j]>
  for (int i = warp; i < Lk; i += CY_WARPS) {
    float acc = 0.f;
    for (int j = 0; j < ch; ++j) {
      const float* kr = K + static_cast<long long>(off + i + j) * C;
      const float* dr = dw + j * C;
      for (int c = lane; c < C; c += 32) acc = fmaf(dr[c], kr[c], acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) dsim[i] = acc;
  }
  __syncthreads();
  if (warp == 0) {
    float dot = 0.f;
    for (int i = lane; i < Lk; i += 32) dot = fmaf(beta[i], dsim[i], dot);
    dot = warp_sum(dot);
    if (lane == 0) bcast = dot;
  }
  __syncthreads();
  {
    const float dot = bcast;
    for (int i = tid; i < Lk; i += CY_THREADS) dsim[i] = beta[i] * (dsim[i] - dot);     // d sim (softmax backward)
  }
  __syncthreads();
  // one (row, channel) element per thread and step, coalesced along the channels
  for (int it = tid; it < T * C; it += CY_THREADS) {
    const int r = it / C, c = it - r * C;
    const float x = feat[it];
    float g = 0.f;
    if (r < R) {
      // query region:  -2a sum_j dz_{r-off-j} (feat[r] - w_j)   [0 <= r-off-j < Lq]
      //                + dq_{r-s}   [0 <= r-s < ch],  dq_j = 2a sum_i dsim_i (K[i+j] - q_j)
      for (int j = 0; j < ch; ++j) {
        const int m = r - off - j;
        if (m >= 0 && m < Lq) g = fmaf(-2.f * a * dz[m], x - w[j * C + c], g);
      }
      const int jq = r - s;
      if (jq >= 0 && jq < ch) {                              // feat[s + jq] is this row: x = q_jq
        const float* kc = K + static_cast<long long>(jq) * C + c;
        float d0 = 0.f, d1 = 0.f;
        int i = 0;
        for (; i + 1 < Lk; i += 2) {
          d0 = fmaf(dsim[i], kc[static_cast<long long>(i) * C] - x, d0);
          d1 = fmaf(dsim[i + 1], kc[static_cast<long long>(i + 1) * C] - x, d1);
        }
        if (i < Lk) d0 = fmaf(dsim[i], kc[static_cast<long long>(i) * C] - x, d0);
        g = fmaf(2.f * a, d0 + d1, g);
      }
    } else {
      // key region, k = r - R:  sum_j beta_{k-off-j} dw_j  [0 <= k-off-j < Lk]  - 2a sum_j dsim_{k-j} (K[k] - q_j)  [0 <= k-j < Lk]
      const int k = r - R;
      for (int j = 0; j < ch; ++j) {
        const int ib = k - off - j, is = k - j;
        if (ib >= 0 && ib < Lk) g = fmaf(beta[ib], dw[j * C + c], g);
        if (is >= 0 && is < Lk) g = fmaf(-2.f * a * dsim[is], x - q[static_cast<long long>(j) * C + c], g);
      }
    }
    part[it] = g;
  }
}

__global__ void cycle_reduce_kernel(const float* __restrict__ part, const float* __restrict__ loss_part, int n_starts,
                                    long long n, float scale, float* __restrict__ dfeat, float* __restrict__ loss) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) {
    float acc = 0.f;
    for (int s = 0; s < n_starts; ++s) acc += part[static_cast<long long>(s) * n + i];
    dfeat[i] = acc * scale;
  }
  if (i == 0) {
    float acc = 0.f;
    for (int s = 0; s < n_starts; ++s) acc += loss_part[s];
    *loss = acc * scale;
  }
}

// ------------------------------------------------------------------------------------------------ spatial sums
// out[b, c] = sum_t x[b, c, t]  for a [B, C, T] view with element strides (sb, sc, st); fp32 accumulation in a fixed
// order.  Channels-last sources (sc == 1, the fusion path's outputs) are read 8 rows at a time, coalesced along C.
template <typename TIn>
__device__ __forceinline__ float cy_ld(const TIn* p);
template <> __device__ __forceinline__ float cy_ld<float>(const float* p) { return *p; }
template <> __device__ __forceinline__ float cy_ld<bf16>(const bf16* p) { return __bfloat162float(*p); }
template <> __device__ __forceinline__ float cy_ld<f16>(const f16* p) { return __half2float(*p); }

template <typename TIn, int VEC>
__device__ __forceinline__ void cy_ld_vec(const TIn* p, float (&f)[VEC]) {
  if constexpr (VEC == 1) {
    f[0] = cy_ld<TIn>(p);
  } else if constexpr (sizeof(TIn) == 2) {                   // 8 bf16 / fp16 = 16 bytes
    const uint4 q = *reinterpret_cast<const uint4*>(p);
    const uint32_t* u = reinterpret_cast<const uint32_t*>(&q);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float2 t;
      if constexpr (std::is_same<TIn, bf16>::value) t = __bfloat1622float2(reinterpret_cast<const __nv_bfloat162*>(u)[j]);
      else t = __half22float2(reinterpret_cast<const __half2*>(u)[j]);
      f[2 * j] = t.x; f[2 * j + 1] = t.y;
    }
  } else {                                                   // 4 fp32 = 16 bytes
    const float4 q = *reinterpret_cast<const float4*>(p);
    f[0] = q.x; f[1] = q.y; f[2] = q.z; f[3] = q.w;
  }
}

template <typename TIn, int VEC>
__global__ void __launch_bounds__(256) spatial_sums_cl_kernel(const TIn* __restrict__ x, long long sb, long long st,
                                                              int C, int T, float* __restrict__ out) {
  __shared__ float red[8][32 * VEC];
  const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
  const int c = (blockIdx.x * 32 + lane) * VEC;
  const TIn* src = x + blockIdx.y * sb + c;
  float acc[VEC];
#pragma unroll
  for (int k = 0; k < VEC; ++k) acc[k] = 0.f;
  if (c < C) {
    int t = grp;
    for (; t + 24 < T; t += 32) {                            // four independent rows in flight per thread
      float f0[VEC], f1[VEC], f2[VEC], f3[VEC];
      cy_ld_vec<TIn, VEC>(src + t * st, f0);
      cy_ld_vec<TIn, VEC>(src + (t + 8) * st, f1);
      cy_ld_vec<TIn, VEC>(src + (t + 16) * st, f2);
      cy_ld_vec<TIn, VEC>(src + (t + 24) * st, f3);
#pragma unroll
      for (int k = 0; k < VEC; ++k) acc[k] += (f0[k] + f1[k]) + (f2[k] + f3[k]);
    }
    for (; t < T; t += 8) {
      float f0[VEC];
      cy_ld_vec<TIn, VEC>(src + t * st, f0);
#pragma unroll
      for (int k = 0; k < VEC; ++k) acc[k] += f0[k];
    }
  }
#pragma unroll
  for (int k = 0; k < VEC; ++k) red[grp][lane * VEC + k] = acc[k];
  __syncthreads();
  for (int i = threadIdx.x; i < 32 * VEC; i += 256) {
    const int cc = blockIdx.x * 32 * VEC + i;
    if (cc < C) {
      float s = 0.f;
#pragma unroll
      for (int g = 0; g < 8; ++g) s += red[g][i];
      out[static_cast<long long>(blockIdx.y) * C + cc] = s;
    }
  }
}

template <typename TIn>
__global__ void __launch_bounds__(256) spatial_sums_any_kernel(const TIn* __restrict__ x, long long sb, long long sc,
                                                               long long st, int C, int T, long long rows,
                                                               float* __restrict__ out) {
  const long long row = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);    // (b, c)
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const TIn* src = x + (row / C) * sb + (row % C) * sc;
  float acc = 0.f;
  for (int t = lane; t < T; t += 32) acc += cy_ld<TIn>(src + t * st);
  acc = warp_sum(acc);
  if (lane == 0) out[row] = acc;
}

}  // namespace

size_t cycle_loss_scratch_bytes(int T, int C, int n_starts) {
  return (static_cast<size_t>(n_starts) * T * C + n_starts) * sizeof(float);
}

int cycle_loss(const float* feat, int T, int C, int R, int off, int ch, float temperature, int start, int step,
               int n_starts, int soft_label, float scale, float* loss, float* dfeat, float* scratch,
               cudaStream_t stream) {
  const int nk = T - R, Lk = nk - ch - off + 1, Lq = R - off - ch + 1;
  if (T <= 0 || C <= 0 || R <= 0 || off < 0 || ch <= 0 || Lk < 1 || Lq < 1)
    return set_error(GLF_ERR_INVALID, "cycle_loss: not enough frames for target_region / cyc_off / chunk_size");
  if (n_starts < 1 || step < 1 || start < 0 || start + (n_starts - 1) * step >= Lq)
    return set_error(GLF_ERR_INVALID, "cycle_loss: start positions outside [0, target_region - chunk_size - cyc_off]");
  if (soft_label && Lq < 2) return set_error(GLF_ERR_INVALID, "cycle_loss: soft labels need two positions");
  if (Lk > CY_MAXPOS || Lq > CY_MAXPOS) return set_error(GLF_ERR_UNSUPPORTED, "cycle_loss: more than 1024 positions");
  const size_t smem = (2 * static_cast<size_t>(ch) * C + 2 * Lk + Lq) * sizeof(float);
  if (smem > 200 * 1024) return set_error(GLF_ERR_UNSUPPORTED, "cycle_loss: chunk_size * C too large for shared memory");
  if (smem > 48 * 1024)
    GLF_TRY(check_cuda(cudaFuncSetAttribute(cycle_start_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            static_cast<int>(smem)), "cycle_loss smem attribute"));
  CycleParams P;
  P.feat = feat; P.T = T; P.C = C; P.R = R; P.off = off; P.ch = ch;
  P.a = temperature / (static_cast<float>(C) * static_cast<float>(ch));
  P.s0 = start; P.step = step; P.n_starts = n_starts; P.soft_label = soft_label;
  P.part = scratch;
  P.loss_part = scratch + static_cast<size_t>(n_starts) * T * C;
  cycle_start_kernel<<<n_starts, CY_THREADS, smem, stream>>>(P);
  GLF_TRY(check_cuda(cudaGetLastError(), "cycle_start launch"));
  const long long n = static_cast<long long>(T) * C;
  cycle_reduce_kernel<<<static_cast<int>((n + 255) / 256), 256, 0, stream>>>(P.part, P.loss_part, n_starts, n, scale,
                                                                             dfeat, loss);
  return check_cuda(cudaGetLastError(), "cycle_reduce launch");
}

int spatial_sums(const void* x, int dtype, int B, int C, int T, long long sb, long long sc, long long st, float* out,
                 cudaStream_t stream) {
  if (B <= 0 || C <= 0 || T <= 0) return set_error(GLF_ERR_INVALID, "spatial_sums: empty input");
  if (dtype != GLF_DTYPE_BF16 && dtype != GLF_DTYPE_F16 && dtype != GLF_DTYPE_F32)
    return set_error(GLF_ERR_INVALID, "spatial_sums: bad dtype");
  if (sc == 1 && B <= 65535) {
    const int per16 = dtype == GLF_DTYPE_F32 ? 4 : 8;
    const bool vec = C % per16 == 0 && sb % per16 == 0 && st % per16 == 0 && reinterpret_cast<uintptr_t>(x) % 16 == 0;
    const dim3 grid((C + 32 * (vec ? per16 : 1) - 1) / (32 * (vec ? per16 : 1)), B);
    if (dtype == GLF_DTYPE_BF16) {
      if (vec) spatial_sums_cl_kernel<bf16, 8><<<grid, 256, 0, stream>>>(reinterpret_cast<const bf16*>(x), sb, st, C, T, out);
      else spatial_sums_cl_kernel<bf16, 1><<<grid, 256, 0, stream>>>(reinterpret_cast<const bf16*>(x), sb, st, C, T, out);
    } else if (dtype == GLF_DTYPE_F16) {
      if (vec) spatial_sums_cl_kernel<f16, 8><<<grid, 256, 0, stream>>>(reinterpret_cast<const f16*>(x), sb, st, C, T, out);
      else spatial_sums_cl_kernel<f16, 1><<<grid, 256, 0, stream>>>(reinterpret_cast<const f16*>(x), sb, st, C, T, out);
    } else {
      if (vec) spatial_sums_cl_kernel<float, 4><<<grid, 256, 0, stream>>>(reinterpret_cast<const float*>(x), sb, st, C, T, out);
      else spatial_sums_cl_kernel<float, 1><<<grid, 256, 0, stream>>>(reinterpret_cast<const float*>(x), sb, st, C, T, out);
    }
  } else {
    const long long rows = static_cast<long long>(B) * C;
    const int grid = static_cast<int>((rows + 7) / 8);
    if (dtype == GLF_DTYPE_BF16)
      spatial_sums_any_kernel<bf16><<<grid, 256, 0, stream>>>(reinterpret_cast<const bf16*>(x), sb, sc, st, C, T, rows, out);
    else if (dtype == GLF_DTYPE_F16)
      spatial_sums_any_kernel<f16><<<grid, 256, 0, stream>>>(reinterpret_cast<const f16*>(x), sb, sc, st, C, T, rows, out);
    else
      spatial_sums_any_kernel<float><<<grid, 256, 0, stream>>>(reinterpret_cast<const float*>(x), sb, sc, st, C, T, rows, out);
  }
  return check_cuda(cudaGetLastError(), "spatial_sums launch");
}

}  // namespace glf
