// glf_eltwise.cu — the HBM-bound kernels of the fusion path: layout packing, weight preparation, BatchNorm
// statistics finalisation, fused BN-normalise + residual + LayerNorm forward/backward, BN-backward apply,
// fp32 -> bf16 casts, partial-sum reductions.
// All row kernels use 128-bit loads/stores, one warp per (row, 256-channel slice), warp-shuffle reductions, and
// per-CTA partials + fixed-order finalisation for every cross-row (per-channel) statistic, so results are
// deterministic (SURVEY.md §7 "hard parts").

#include <type_traits>

#include "glf_internal.h"
#include "glf_ptx.cuh"

namespace glf {

namespace {

constexpr int ROW_THREADS = 256;
constexpr int ROW_WARPS = ROW_THREADS / 32;

__device__ __forceinline__ void load8(const bf16* p, float (&f)[8]) {
  const uint4 v = *reinterpret_cast<const uint4*>(p);
  const uint32_t* u = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = unpack_bf16(u[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ void load8(const f16* p, float (&f)[8]) {
  const uint4 v = *reinterpret_cast<const uint4*>(p);
  const uint32_t* u = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = unpack2<f16>(u[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ void load8(const float* p, float (&f)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p);
  const float4 b = *reinterpret_cast<const float4*>(p + 4);
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w;
  f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}
__device__ __forceinline__ void store8(bf16* p, const float (&f)[8]) {
  uint4 v = make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
  *reinterpret_cast<uint4*>(p) = v;
}
__device__ __forceinline__ void store8(f16* p, const float (&f)[8]) {
  uint4 v = make_uint4(pack2<f16>(f[0], f[1]), pack2<f16>(f[2], f[3]), pack2<f16>(f[4], f[5]), pack2<f16>(f[6], f[7]));
  *reinterpret_cast<uint4*>(p) = v;
}
__device__ __forceinline__ void store8(float* p, const float (&f)[8]) {
  *reinterpret_cast<float4*>(p) = make_float4(f[0], f[1], f[2], f[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(f[4], f[5], f[6], f[7]);
}

// Sum over the S warps that share one row (slices of 256 channels). red: [2][ROW_WARPS] floats, `buf` alternates.
template <int NV>
__device__ __forceinline__ void row_reduce(float (&v)[NV], int S, int rslot, int slice, float* red, int& buf) {
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = warp_sum(v[i]);
  if (S > 1) {
    float* r = red + buf * (ROW_WARPS * NV);
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
      for (int i = 0; i < NV; ++i) r[(rslot * S + slice) * NV + i] = v[i];
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      float s = 0.f;
      for (int j = 0; j < S; ++j) s += r[(rslot * S + j) * NV + i];
      v[i] = s;
    }
    buf ^= 1;
  }
}

// ------------------------------------------------------------------------------------------------ transpose + cast
template <typename TI, typename TO>
__global__ void transpose_kernel(const TI* __restrict__ in, TO* __restrict__ out, int R, int S) {
  __shared__ float tile[64][65];
  const long long boff = static_cast<long long>(blockIdx.z) * R * S;
  const int r0 = blockIdx.y * 64, s0 = blockIdx.x * 64;
  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;  // 64 x 4
  for (int i = ty; i < 64; i += 4) {
    const int r = r0 + i, s = s0 + tx;
    if (r < R && s < S) tile[i][tx] = static_cast<float>(in[boff + static_cast<long long>(r) * S + s]);
  }
  __syncthreads();
  for (int j = ty; j < 64; j += 4) {
    const int s = s0 + j, r = r0 + tx;
    if (r < R && s < S) out[boff + static_cast<long long>(s) * R + r] = static_cast<TO>(tile[tx][j]);
  }
}

// ------------------------------------------------------------------------------------------------ weights
// fp32 masters -> bf16 operands: Wcat [3Ci, C] (theta | phi | g), WcatT [C, 3Ci], bcat [3Ci] fp32, Wz [C, Ci], WzT [Ci, C]
// 32 x 32 tiles, transposed through shared memory: every global access is coalesced (the element-per-thread version
// spent 80 us at C = 2048 on its strided transposed stores).
__global__ void __launch_bounds__(256) prep_weights_kernel(const float* __restrict__ tw, const float* __restrict__ pw,
                                    const float* __restrict__ gw, const float* __restrict__ tb,
                                    const float* __restrict__ pb, const float* __restrict__ gb,
                                    const float* __restrict__ wz, bf16* __restrict__ wcat, bf16* __restrict__ wcatT,
                                    float* __restrict__ bcat, bf16* __restrict__ wzb, bf16* __restrict__ wzT, int C,
                                    int Ci) {
  __shared__ float tile[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;       // 32 x 8
  const int tc = (C + 31) / 32, tci = (Ci + 31) / 32;
  const int n_cat = 3 * tci * tc;                                // tiles of Wcat: rows 3Ci (tile rows never straddle a projection)
  int t = blockIdx.x;
  const float* src; bf16* dst; bf16* dstT;
  int R, Cc, r0, c0;                                             // source [R, Cc] row-major; destination row offset for the concatenation
  long long dst_ld, dstT_ld; int dst_row_off;
  if (t < n_cat) {
    const int which = t / (tci * tc), rem = t % (tci * tc);
    src = which == 0 ? tw : (which == 1 ? pw : gw);
    R = Ci; Cc = C; r0 = (rem / tc) * 32; c0 = (rem % tc) * 32;
    dst = wcat; dst_ld = C; dstT = wcatT; dstT_ld = 3LL * Ci; dst_row_off = which * Ci;
  } else {
    t -= n_cat;
    src = wz; R = C; Cc = Ci; r0 = (t / tci) * 32; c0 = (t % tci) * 32;
    dst = wzb; dst_ld = Ci; dstT = wzT; dstT_ld = C; dst_row_off = 0;
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = r0 + ty + 8 * i, c = c0 + tx;
    float v = 0.f;
    if (r < R && c < Cc) {
      v = src[static_cast<long long>(r) * Cc + c];
      dst[static_cast<long long>(dst_row_off + r) * dst_ld + c] = __float2bfloat16(v);
    }
    tile[ty + 8 * i][tx] = v;
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = c0 + ty + 8 * i, r = r0 + tx;                  // transposed: row c of the destination, column (offset + r)
    if (r < R && c < Cc) dstT[static_cast<long long>(c) * dstT_ld + dst_row_off + r] = __float2bfloat16(tile[tx][ty + 8 * i]);
  }
  if (blockIdx.x == 0)
    for (int i = threadIdx.x; i < 3 * Ci; i += 256) {
      const int w2 = i / Ci, k = i % Ci;
      bcat[i] = (w2 == 0 ? tb : (w2 == 1 ? pb : gb))[k];
    }
}

// ------------------------------------------------------------------------------------------------ BN statistics
// Block = 32 channels x RED_Y partial groups.  Every thread sums a strided subset of the partial rows in double,
// the RED_Y sub-sums are combined through shared memory in a fixed order -> deterministic, no atomics.
constexpr int RED_Y = 32;
template <int NS>
__device__ __forceinline__ void reduce_partial_rows(const float* __restrict__ part, int np, long long row_stride,
                                                    long long stat_stride, int c, bool cact, double (&out)[NS],
                                                    double (*sm)[RED_Y][33]) {
  double acc[NS];
#pragma unroll
  for (int j = 0; j < NS; ++j) acc[j] = 0.0;
  if (cact) {
    // four independent partial sums per statistic keep four loads in flight; combined in a fixed order
    double a4[NS][4];
#pragma unroll
    for (int j = 0; j < NS; ++j) a4[j][0] = a4[j][1] = a4[j][2] = a4[j][3] = 0.0;
    int i = threadIdx.y;
    for (; i + 3 * RED_Y < np; i += 4 * RED_Y) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
#pragma unroll
        for (int j = 0; j < NS; ++j)
          a4[j][u] += static_cast<double>(part[(i + u * RED_Y) * row_stride + j * stat_stride + c]);
      }
    }
    for (; i < np; i += RED_Y) {
#pragma unroll
      for (int j = 0; j < NS; ++j) a4[j][0] += static_cast<double>(part[i * row_stride + j * stat_stride + c]);
    }
#pragma unroll
    for (int j = 0; j < NS; ++j) acc[j] = (a4[j][0] + a4[j][1]) + (a4[j][2] + a4[j][3]);
  }
#pragma unroll
  for (int j = 0; j < NS; ++j) sm[j][threadIdx.y][threadIdx.x] = acc[j];
  __syncthreads();
#pragma unroll
  for (int j = 0; j < NS; ++j) {
    double t = 0.0;
    for (int y = 0; y < RED_Y; ++y) t += sm[j][y][threadIdx.x];
    out[j] = t;
  }
}

// Stage 1 of the two-stage reductions: G row-slices of the partial table are reduced by G x (C/32) CTAs in parallel
// (fixed order inside every slice); the finalisers then combine G rows.  Up to 3 tables per launch (blockIdx.z).
struct Stage1 {
  const float* part[3];
  float* out[3];          // [G][NS][C]
  int np[3];              // rows of each table
};
template <int NS>
__global__ void __launch_bounds__(32 * RED_Y)
    reduce_stage1_kernel(const Stage1 t, long long row_stride, long long stat_stride, int C, int G) {
  __shared__ double sm[NS][RED_Y][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const bool cact = c < C;
  const int g = blockIdx.y;
  const int np = t.np[blockIdx.z];
  const int chunk = (np + G - 1) / G;
  const int r0 = g * chunk;
  const int cnt = max(0, min(np, r0 + chunk) - r0);
  double s[NS];
  reduce_partial_rows<NS>(t.part[blockIdx.z] + static_cast<long long>(r0) * row_stride, cnt, row_stride, stat_stride, c,
                          cact, s, sm);
  if (threadIdx.y == 0 && cact) {
#pragma unroll
    for (int j = 0; j < NS; ++j) t.out[blockIdx.z][(static_cast<long long>(g) * NS + j) * C + c] = static_cast<float>(s[j]);
  }
}

// running statistics in the parameters' element type, updated in fp64 and rounded once
__device__ __forceinline__ double ld_stat(const float* p) { return *p; }
__device__ __forceinline__ double ld_stat(const bf16* p) { return __bfloat162float(*p); }
__device__ __forceinline__ double ld_stat(const f16* p) { return __half2float(*p); }
__device__ __forceinline__ void st_stat(float* p, double v) { *p = static_cast<float>(v); }
__device__ __forceinline__ void st_stat(bf16* p, double v) { *p = __double2bfloat16(v); }
__device__ __forceinline__ void st_stat(f16* p, double v) { *p = __double2half(v); }

// partials: [np][2][C] (sum, sum of squares) -> mean, rstd, affine a = gamma*rstd, b = beta - mean*a; running stats.
template <typename TR>
__global__ void __launch_bounds__(32 * RED_Y)
    bn_finalize_kernel(const float* __restrict__ part, int np, int C, double count, const float* __restrict__ gamma,
                       const float* __restrict__ beta, const float* __restrict__ bz, float eps, float momentum,
                       int training, int bn_layer,
                       TR* __restrict__ rm, TR* __restrict__ rv, long long* __restrict__ nbt,
                       float* __restrict__ mean_o, float* __restrict__ rstd_o, float* __restrict__ a_o,
                       float* __restrict__ b_o) {
  __shared__ double sm[2][RED_Y][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const bool cact = c < C;
  double st[2] = {0.0, 0.0};
  if (training && bn_layer) reduce_partial_rows<2>(part, np, 2LL * C, C, c, cact, st, sm);
  if (threadIdx.y != 0 || !cact) return;
  if (c == 0 && training && bn_layer && nbt != nullptr) *nbt += 1;
  // bz != nullptr: the W_z bias was NOT added to the stored U (train-mode BatchNorm cancels it, so the GEMM epilogue
  // skips the add); it is folded into the affine here and restored in the running mean
  const double shift = bz != nullptr ? static_cast<double>(bz[c]) : 0.0;
  if (!bn_layer) {
    mean_o[c] = 0.f; rstd_o[c] = 1.f; a_o[c] = 1.f; b_o[c] = static_cast<float>(shift);
    return;
  }
  double mean, var;
  if (training) {
    mean = st[0] / count;
    var = st[1] / count - mean * mean;
    if (var < 0.0) var = 0.0;
    const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
    st_stat(rm + c, (1.0 - momentum) * ld_stat(rm + c) + momentum * (mean + shift));
    st_stat(rv + c, (1.0 - momentum) * ld_stat(rv + c) + momentum * unbiased);
  } else {
    mean = ld_stat(rm + c) - shift;
    var = ld_stat(rv + c);
  }
  const double rstd = 1.0 / sqrt(var + static_cast<double>(eps));
  const double a = gamma[c] * rstd;
  mean_o[c] = static_cast<float>(mean);
  rstd_o[c] = static_cast<float>(rstd);
  a_o[c] = static_cast<float>(a);
  b_o[c] = static_cast<float>(beta[c] - mean * a);
}

// ------------------------------------------------------------------------------------------------ BN + residual + LN fwd
// Raw (still packed) 8-element vectors: the next row is fetched while the current one is processed, which doubles
// the bytes in flight per warp (the kernels are latency-bound on HBM otherwise: ~45 % of peak measured without it).
template <typename T> struct Raw8;
template <> struct Raw8<bf16> { uint4 v; };
template <> struct Raw8<f16> { uint4 v; };
template <> struct Raw8<float> { float4 a, b; };
__device__ __forceinline__ Raw8<bf16> ldraw(const bf16* p) {
  Raw8<bf16> r;
  r.v = *reinterpret_cast<const uint4*>(p);
  return r;
}
__device__ __forceinline__ Raw8<f16> ldraw(const f16* p) {
  Raw8<f16> r;
  r.v = *reinterpret_cast<const uint4*>(p);
  return r;
}
__device__ __forceinline__ Raw8<float> ldraw(const float* p) {
  Raw8<float> r;
  r.a = *reinterpret_cast<const float4*>(p);
  r.b = *reinterpret_cast<const float4*>(p + 4);
  return r;
}
__device__ __forceinline__ void cvt8(const Raw8<bf16>& r, float (&f)[8]) {
  const uint32_t* u = reinterpret_cast<const uint32_t*>(&r.v);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = unpack_bf16(u[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ void cvt8(const Raw8<f16>& r, float (&f)[8]) {
  const uint32_t* u = reinterpret_cast<const uint32_t*>(&r.v);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = unpack2<f16>(u[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ void cvt8(const Raw8<float>& r, float (&f)[8]) {
  f[0] = r.a.x; f[1] = r.a.y; f[2] = r.a.z; f[3] = r.a.w;
  f[4] = r.b.x; f[5] = r.b.y; f[6] = r.b.z; f[7] = r.b.w;
}

// volatile 2 x 128-bit shared-memory load (keeps loop-invariant vectors out of the register file)
__device__ __forceinline__ void lds8v(const float* p, float (&f)[8]) {
  const uint32_t a = smem_u32(p);
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(f[0]), "=f"(f[1]), "=f"(f[2]), "=f"(f[3]) : "r"(a));
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(f[4]), "=f"(f[5]), "=f"(f[6]), "=f"(f[7])
               : "r"(a + 16));
}

// Z = LayerNorm_C(a*U + b + X) * lw + lb     (ours.py:908-915 after the W_z GEMM).  U may be nullptr (V = 0).
template <typename TO, typename TA>
__global__ void __launch_bounds__(ROW_THREADS)
    bn_res_ln_fwd_kernel(const TA* __restrict__ U, const TA* __restrict__ X, const float* __restrict__ bn_a,
                         const float* __restrict__ bn_b, const float* __restrict__ lw, const float* __restrict__ lb,
                         TO* __restrict__ Z, float* __restrict__ mu_o, float* __restrict__ r_o, long long rows, int C,
                         int S, float eps, int accumulate) {
  __shared__ float red[2 * ROW_WARPS * 2];
  int buf = 0;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int RPB = ROW_WARPS / S;
  const int rslot = warp / S, slice = warp % S;
  const int c0 = slice * 256 + lane * 8;
  const bool cact = c0 < C;
  float a[8], b[8], w[8], bb[8];
  if (cact) {
    load8(bn_a + c0, a); load8(bn_b + c0, b); load8(lw + c0, w); load8(lb + c0, bb);
  }
  const float invC = 1.f / static_cast<float>(C);
  const long long step = static_cast<long long>(gridDim.x) * RPB;
  long long base = static_cast<long long>(blockIdx.x) * RPB;
  Raw8<TA> xr = {}, ur = {};
  if (cact && base + rslot < rows) {
    xr = ldraw(X + (base + rslot) * C + c0);
    if (U != nullptr) ur = ldraw(U + (base + rslot) * C + c0);
  }
  for (; base < rows; base += step) {
    const long long row = base + rslot;
    const bool act = cact && row < rows;
    const Raw8<TA> xc = xr, uc = ur;
    if (cact && row + step < rows) {
      xr = ldraw(X + (row + step) * C + c0);
      if (U != nullptr) ur = ldraw(U + (row + step) * C + c0);
    }
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = 0.f;
    if (act) {
      float x[8];
      cvt8(xc, x);
      if (U != nullptr) {
        float u[8];
        cvt8(uc, u);
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = fmaf(a[i], u[i], b[i]) + x[i];
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = x[i];
      }
    }
    float s[1] = {0.f};
#pragma unroll
    for (int i = 0; i < 8; ++i) s[0] += v[i];
    row_reduce<1>(s, S, rslot, slice, red, buf);
    const float mu = s[0] * invC;
    float q[1] = {0.f};
    if (act) {
#pragma unroll
      for (int i = 0; i < 8; ++i) q[0] = fmaf(v[i] - mu, v[i] - mu, q[0]);
    }
    row_reduce<1>(q, S, rslot, slice, red, buf);
    const float r = rsqrtf(q[0] * invC + eps);
    if (act) {
      float o[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = fmaf((v[i] - mu) * r, w[i], bb[i]);
      if (accumulate) {
        float z0[8];
        load8(Z + row * C + c0, z0);
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] += z0[i];
      }
      store8(Z + row * C + c0, o);
      if (slice == 0 && lane == 0 && mu_o != nullptr) {
        mu_o[row] = mu;
        r_o[row] = r;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ BN + residual + LN bwd
// From dZ: dV = dZp (gradient of the pre-LayerNorm sum, also the residual part of dX), and per-CTA partials of the
// four per-channel reductions: d ln_w = sum dZ*xhat, d ln_b = sum dZ, d gamma = sum dV*uhat, d beta = sum dV.
template <typename TI, typename TA>
__global__ void __launch_bounds__(ROW_THREADS, 2)
    bn_res_ln_bwd_kernel(const TI* __restrict__ dZ, const TA* __restrict__ U, const TA* __restrict__ X,
                         const float* __restrict__ bn_a, const float* __restrict__ bn_b,
                         const float* __restrict__ bn_mean, const float* __restrict__ bn_rstd,
                         const float* __restrict__ lw, const float* __restrict__ mu_i, const float* __restrict__ r_i,
                         TA* __restrict__ dV, float* __restrict__ part, long long rows, int C, int S) {
  __shared__ float red[2 * ROW_WARPS * 2];
  // per-channel parameter vectors live in shared memory during the row loop (re-read with volatile 128-bit loads so
  // that they do not occupy 40 registers); the same storage holds the accumulator exchange afterwards
  constexpr int ACC_PITCH = 32 * 8 + 8;
  constexpr int SM_FLOATS = (ROW_WARPS * 4 * ACC_PITCH > 5 * 2048) ? ROW_WARPS * 4 * ACC_PITCH : 5 * 2048;
  __shared__ __align__(16) float smbuf[SM_FLOATS];
  int buf = 0;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int RPB = ROW_WARPS / S;
  const int rslot = warp / S, slice = warp % S;
  const int c0 = slice * 256 + lane * 8;
  const bool cact = c0 < C;
  const int Cs = S * 256;
  for (int i = threadIdx.x; i < Cs; i += ROW_THREADS) {
    const bool in = i < C;
    smbuf[0 * Cs + i] = in ? bn_a[i] : 0.f;
    smbuf[1 * Cs + i] = in ? bn_b[i] : 0.f;
    smbuf[2 * Cs + i] = in ? lw[i] : 0.f;
    smbuf[3 * Cs + i] = in ? bn_mean[i] : 0.f;
    smbuf[4 * Cs + i] = in ? bn_rstd[i] : 0.f;
  }
  __syncthreads();
  const float* sp = smbuf + c0;
  float g_lw[8], g_lb[8], g_ga[8], g_be[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) g_lw[i] = g_lb[i] = g_ga[i] = g_be[i] = 0.f;
  const float invC = 1.f / static_cast<float>(C);
  const long long step = static_cast<long long>(gridDim.x) * RPB;
  long long base = static_cast<long long>(blockIdx.x) * RPB;
  Raw8<TA> xr = {}, ur = {};
  Raw8<TI> zr = {};
  float mu_n = 0.f, r_n = 0.f;
  if (cact && base + rslot < rows) {
    const long long row = base + rslot;
    xr = ldraw(X + row * C + c0);
    zr = ldraw(dZ + row * C + c0);
    if (U != nullptr) ur = ldraw(U + row * C + c0);
    mu_n = mu_i[row];
    r_n = r_i[row];
  }
  for (; base < rows; base += step) {
    const long long row = base + rslot;
    const bool act = cact && row < rows;
    const Raw8<TA> xc = xr, uc = ur;
    const Raw8<TI> zc = zr;
    const float mu = mu_n, r = r_n;
    if (cact && row + step < rows) {
      const long long nrow = row + step;
      xr = ldraw(X + nrow * C + c0);
      zr = ldraw(dZ + nrow * C + c0);
      if (U != nullptr) ur = ldraw(U + nrow * C + c0);
      mu_n = mu_i[nrow];
      r_n = r_i[nrow];
    }
    float xh[8], dxh[8], dz[8], uh[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) xh[i] = dxh[i] = dz[i] = uh[i] = 0.f;
    if (act) {
      float x[8];
      cvt8(xc, x);
      cvt8(zc, dz);
      if (U != nullptr) {
        float u[8], a[8], b[8];
        cvt8(uc, u);
        lds8v(sp, a);
        lds8v(sp + Cs, b);
#pragma unroll
        for (int i = 0; i < 8; ++i) xh[i] = (fmaf(a[i], u[i], b[i]) + x[i] - mu) * r;
        lds8v(sp + 3 * Cs, a);
        lds8v(sp + 4 * Cs, b);
#pragma unroll
        for (int i = 0; i < 8; ++i) uh[i] = (u[i] - a[i]) * b[i];
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) xh[i] = (x[i] - mu) * r;
      }
      float w[8];
      lds8v(sp + 2 * Cs, w);
#pragma unroll
      for (int i = 0; i < 8; ++i) dxh[i] = dz[i] * w[i];
    }
    float s[2] = {0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      s[0] += dxh[i];
      s[1] = fmaf(dxh[i], xh[i], s[1]);
    }
    row_reduce<2>(s, S, rslot, slice, red, buf);
    if (act) {
      const float m1 = s[0] * invC, m2 = s[1] * invC;
      float dv[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        dv[i] = r * (dxh[i] - m1 - xh[i] * m2);
        g_lw[i] = fmaf(dz[i], xh[i], g_lw[i]);
        g_lb[i] += dz[i];
        g_ga[i] = fmaf(dv[i], uh[i], g_ga[i]);
        g_be[i] += dv[i];
      }
      store8(dV + row * C + c0, dv);
    }
  }
  // reduce the accumulators over the row slots of this CTA (fixed order), write one partial per CTA
  __syncthreads();  // every warp is done with the parameter vectors: reuse the storage
  float (*acc_sm)[4][ACC_PITCH] = reinterpret_cast<float (*)[4][ACC_PITCH]>(smbuf);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    acc_sm[warp][0][lane * 8 + i] = g_lw[i];
    acc_sm[warp][1][lane * 8 + i] = g_lb[i];
    acc_sm[warp][2][lane * 8 + i] = g_ga[i];
    acc_sm[warp][3][lane * 8 + i] = g_be[i];
  }
  __syncthreads();
  // output index space: 4 stats x (S*256) channels
  for (int idx = threadIdx.x; idx < 4 * S * 256; idx += ROW_THREADS) {
    const int st = idx / (S * 256), cc = idx % (S * 256);
    const int sl = cc / 256, ci = cc % 256;
    if (cc < C) {
      float t = 0.f;
      for (int rs = 0; rs < RPB; ++rs) t += acc_sm[rs * S + sl][st][ci];
      part[(static_cast<long long>(blockIdx.x) * 4 + st) * C + cc] = t;
    }
  }
}

// ------------------------------------------------------------------------------------------------ wide rows (C > 256)
// Rows wider than 256 channels are sliced over S warps, so a CTA of 8 warps holds one or two rows per step and the
// register-prefetch kernels above keep ~48 KB per SM in flight: 2.7 - 3.7 TB/s at C = 2048.  (More rows per thread was
// tried: 139 registers, one CTA per SM, slower.)  These bf16 variants prefetch through a per-thread ring in shared memory
// instead: every thread issues 16-byte cp.async copies LN_DEPTH - 1 steps ahead into slots only it reads back, so there
// is nothing to synchronise beyond cp.async.wait_group and the depth costs no registers.
constexpr int LN_DEPTH = 4;

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ring layout: [LN_DEPTH][nops][ROW_THREADS] uint4.  TZ: bf16 or fp16 Z (same bytes per row).
template <typename TZ>
__global__ void __launch_bounds__(ROW_THREADS)
    bn_res_ln_fwd_ring_kernel(const bf16* __restrict__ U, const bf16* __restrict__ X, const float* __restrict__ bn_a,
                              const float* __restrict__ bn_b, const float* __restrict__ lw, const float* __restrict__ lb,
                              TZ* __restrict__ Z, float* __restrict__ mu_o, float* __restrict__ r_o, long long rows, int C,
                              int S, float eps, int accumulate) {
  extern __shared__ __align__(16) uint4 ln_ring[];
  __shared__ float red[2 * ROW_WARPS * 2];
  int buf = 0;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int RPB = ROW_WARPS / S;
  const int rslot = warp / S, slice = warp % S;
  const int c0 = slice * 256 + lane * 8;
  const bool cact = c0 < C;
  float a[8], b[8], w[8], bb[8];
  if (cact) {
    load8(bn_a + c0, a); load8(bn_b + c0, b); load8(lw + c0, w); load8(lb + c0, bb);
  }
  const float invC = 1.f / static_cast<float>(C);
  const long long step = static_cast<long long>(gridDim.x) * RPB;
  const long long first = static_cast<long long>(blockIdx.x) * RPB + rslot;
  uint4* mine = ln_ring + threadIdx.x;
  auto issue = [&](long long row, int slot) {
    if (cact && row < rows) {
      uint4* dst = mine + slot * 3 * ROW_THREADS;
      cp_async16(dst, X + row * C + c0);
      if (U != nullptr) cp_async16(dst + ROW_THREADS, U + row * C + c0);
      if (accumulate) cp_async16(dst + 2 * ROW_THREADS, Z + row * C + c0);
    }
    cp_async_commit();
  };
#pragma unroll
  for (int d = 0; d < LN_DEPTH - 1; ++d) issue(first + d * step, d);
  int it = 0;
  for (long long base = static_cast<long long>(blockIdx.x) * RPB; base < rows; base += step, ++it) {
    const long long row = base + rslot;
    const bool act = cact && row < rows;
    issue(row + (LN_DEPTH - 1) * step, (it + LN_DEPTH - 1) % LN_DEPTH);
    cp_async_wait<LN_DEPTH - 1>();
    const uint4* src = mine + (it % LN_DEPTH) * 3 * ROW_THREADS;
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = 0.f;
    if (act) {
      Raw8<bf16> xc, uc;
      xc.v = src[0];
      float x[8];
      cvt8(xc, x);
      if (U != nullptr) {
        uc.v = src[ROW_THREADS];
        float u[8];
        cvt8(uc, u);
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = fmaf(a[i], u[i], b[i]) + x[i];
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = x[i];
      }
    }
    float sm1[1] = {0.f};
#pragma unroll
    for (int i = 0; i < 8; ++i) sm1[0] += v[i];
    row_reduce<1>(sm1, S, rslot, slice, red, buf);
    const float mu = sm1[0] * invC;
    float q[1] = {0.f};
    if (act) {
#pragma unroll
      for (int i = 0; i < 8; ++i) q[0] = fmaf(v[i] - mu, v[i] - mu, q[0]);
    }
    row_reduce<1>(q, S, rslot, slice, red, buf);
    const float r = rsqrtf(q[0] * invC + eps);
    if (act) {
      float o[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = fmaf((v[i] - mu) * r, w[i], bb[i]);
      if (accumulate) {
        Raw8<TZ> zc;
        zc.v = src[2 * ROW_THREADS];
        float z0[8];
        cvt8(zc, z0);
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] += z0[i];
      }
      store8(Z + row * C + c0, o);
      if (slice == 0 && lane == 0 && mu_o != nullptr) {
        mu_o[row] = mu;
        r_o[row] = r;
      }
    }
  }
  cp_async_wait<0>();
}

// The MGFM + MLFM pair of the fused call site for wide rows: Z = sum_m LayerNorm(a_m U_m + b_m + X_m) lw_m + lb_m in ONE pass
// (the two single-block calls read and re-write Z in between: 7 row streams instead of 5), optionally storing module 0's
// own output (f4_global_fusion) as well.  Same slicing and per-thread cp.async ring as bn_res_ln_fwd_ring_kernel.
struct LnPairWide {
  const bf16* U[2];
  const bf16* X[2];
  const float* a[2];
  const float* b[2];
  const float* lw[2];
  const float* lb[2];
  float* mu[2];
  float* r[2];
  void* Z;         // [rows, C] of the kernel's TZ (bf16 or fp16), like Z0
  void* Z0;
  long long rows;
  int C, S, accumulate;
  float eps;
};

template <bool PARTS, typename TZ>
__global__ void __launch_bounds__(ROW_THREADS, 2) ln_pair_fwd_ring_kernel(const LnPairWide p) {
  extern __shared__ __align__(16) uint4 ln_ring[];
  __shared__ float red[2 * ROW_WARPS * 2];
  int buf = 0;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int S = p.S, C = p.C;
  const int RPB = ROW_WARPS / S;
  const int rslot = warp / S, slice = warp % S;
  const int c0 = slice * 256 + lane * 8;
  const bool cact = c0 < C;
  float a0[8], b0[8], w0[8], a1[8], b1[8], w1[8], lbs[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) a0[i] = b0[i] = w0[i] = a1[i] = b1[i] = w1[i] = lbs[i] = 0.f;
  if (cact) {
    float t[8];
    load8(p.a[0] + c0, a0); load8(p.b[0] + c0, b0); load8(p.lw[0] + c0, w0);
    load8(p.a[1] + c0, a1); load8(p.b[1] + c0, b1); load8(p.lw[1] + c0, w1);
    load8(p.lb[0] + c0, lbs); load8(p.lb[1] + c0, t);
    if (!PARTS) {
#pragma unroll
      for (int i = 0; i < 8; ++i) lbs[i] += t[i];             // both biases at once
    }
  }
  const float invC = 1.f / static_cast<float>(C);
  const long long rows = p.rows;
  const long long step = static_cast<long long>(gridDim.x) * RPB;
  const long long first = static_cast<long long>(blockIdx.x) * RPB + rslot;
  uint4* mine = ln_ring + threadIdx.x;
  constexpr int NOPS = 5;
  auto issue = [&](long long row, int slot) {
    if (cact && row < rows) {
      uint4* dst = mine + slot * NOPS * ROW_THREADS;
      const long long off = row * C + c0;
      cp_async16(dst, p.X[0] + off);
      cp_async16(dst + ROW_THREADS, p.U[0] + off);
      cp_async16(dst + 2 * ROW_THREADS, p.X[1] + off);
      cp_async16(dst + 3 * ROW_THREADS, p.U[1] + off);
      if (p.accumulate) cp_async16(dst + 4 * ROW_THREADS, reinterpret_cast<const TZ*>(p.Z) + off);
    }
    cp_async_commit();
  };
#pragma unroll
  for (int d = 0; d < LN_DEPTH - 1; ++d) issue(first + d * step, d);
  int it = 0;
  for (long long base = static_cast<long long>(blockIdx.x) * RPB; base < rows; base += step, ++it) {
    const long long row = base + rslot;
    const bool act = cact && row < rows;
    issue(row + (LN_DEPTH - 1) * step, (it + LN_DEPTH - 1) % LN_DEPTH);
    cp_async_wait<LN_DEPTH - 1>();
    const uint4* src = mine + (it % LN_DEPTH) * NOPS * ROW_THREADS;
    float v0[8], v1[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v0[i] = v1[i] = 0.f;
    if (act) {
      Raw8<bf16> q;
      float x[8], u[8];
      q.v = src[0]; cvt8(q, x);
      q.v = src[ROW_THREADS]; cvt8(q, u);
#pragma unroll
      for (int i = 0; i < 8; ++i) v0[i] = fmaf(a0[i], u[i], b0[i]) + x[i];
      q.v = src[2 * ROW_THREADS]; cvt8(q, x);
      q.v = src[3 * ROW_THREADS]; cvt8(q, u);
#pragma unroll
      for (int i = 0; i < 8; ++i) v1[i] = fmaf(a1[i], u[i], b1[i]) + x[i];
    }
    float sm2[2] = {0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 8; ++i) { sm2[0] += v0[i]; sm2[1] += v1[i]; }
    row_reduce<2>(sm2, S, rslot, slice, red, buf);
    const float mu0 = sm2[0] * invC, mu1 = sm2[1] * invC;
    float q2[2] = {0.f, 0.f};
    if (act) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        q2[0] = fmaf(v0[i] - mu0, v0[i] - mu0, q2[0]);
        q2[1] = fmaf(v1[i] - mu1, v1[i] - mu1, q2[1]);
      }
    }
    row_reduce<2>(q2, S, rslot, slice, red, buf);
    const float r0 = rsqrtf(q2[0] * invC + p.eps), r1 = rsqrtf(q2[1] * invC + p.eps);
    if (act) {
      float o[8];
      if (PARTS) {
        float o0[8], lb1[8];
        load8(p.lb[1] + c0, lb1);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          o0[i] = fmaf((v0[i] - mu0) * r0, w0[i], lbs[i]);
          o[i] = o0[i] + fmaf((v1[i] - mu1) * r1, w1[i], lb1[i]);
        }
        store8(reinterpret_cast<TZ*>(p.Z0) + row * C + c0, o0);
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = fmaf((v0[i] - mu0) * r0, w0[i], fmaf((v1[i] - mu1) * r1, w1[i], lbs[i]));
      }
      if (p.accumulate) {
        Raw8<TZ> zc;
        zc.v = src[4 * ROW_THREADS];
        float z0[8];
        cvt8(zc, z0);
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] += z0[i];
      }
      store8(reinterpret_cast<TZ*>(p.Z) + row * C + c0, o);
      if (slice == 0 && lane == 0) {
        if (p.mu[0] != nullptr) { p.mu[0][row] = mu0; p.r[0][row] = r0; }
        if (p.mu[1] != nullptr) { p.mu[1][row] = mu1; p.r[1][row] = r1; }
      }
    }
  }
  cp_async_wait<0>();
}

template <typename TZ>
__global__ void __launch_bounds__(ROW_THREADS, 2)
    bn_res_ln_bwd_ring_kernel(const TZ* __restrict__ dZ, const bf16* __restrict__ U, const bf16* __restrict__ X,
                              const float* __restrict__ bn_a, const float* __restrict__ bn_b,
                              const float* __restrict__ bn_mean, const float* __restrict__ bn_rstd,
                              const float* __restrict__ lw, const float* __restrict__ mu_i, const float* __restrict__ r_i,
                              bf16* __restrict__ dV, float* __restrict__ part, long long rows, int C, int S) {
  extern __shared__ __align__(16) uint4 ln_ring[];
  __shared__ float red[2 * ROW_WARPS * 2];
  constexpr int ACC_PITCH = 32 * 8 + 8;
  constexpr int SM_FLOATS = (ROW_WARPS * 4 * ACC_PITCH > 5 * 2048) ? ROW_WARPS * 4 * ACC_PITCH : 5 * 2048;
  __shared__ __align__(16) float smbuf[SM_FLOATS];
  int buf = 0;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int RPB = ROW_WARPS / S;
  const int rslot = warp / S, slice = warp % S;
  const int c0 = slice * 256 + lane * 8;
  const bool cact = c0 < C;
  const int Cs = S * 256;
  for (int i = threadIdx.x; i < Cs; i += ROW_THREADS) {
    const bool in = i < C;
    smbuf[0 * Cs + i] = in ? bn_a[i] : 0.f;
    smbuf[1 * Cs + i] = in ? bn_b[i] : 0.f;
    smbuf[2 * Cs + i] = in ? lw[i] : 0.f;
    smbuf[3 * Cs + i] = in ? bn_mean[i] : 0.f;
    smbuf[4 * Cs + i] = in ? bn_rstd[i] : 0.f;
  }
  __syncthreads();
  const float* sp = smbuf + c0;
  float g_lw[8], g_lb[8], g_ga[8], g_be[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) g_lw[i] = g_lb[i] = g_ga[i] = g_be[i] = 0.f;
  const float invC = 1.f / static_cast<float>(C);
  const long long step = static_cast<long long>(gridDim.x) * RPB;
  const long long first = static_cast<long long>(blockIdx.x) * RPB + rslot;
  uint4* mine = ln_ring + threadIdx.x;
  auto issue = [&](long long row, int slot) {
    if (cact && row < rows) {
      uint4* dst = mine + slot * 3 * ROW_THREADS;
      cp_async16(dst, X + row * C + c0);
      cp_async16(dst + ROW_THREADS, dZ + row * C + c0);
      if (U != nullptr) cp_async16(dst + 2 * ROW_THREADS, U + row * C + c0);
    }
    cp_async_commit();
  };
#pragma unroll
  for (int d = 0; d < LN_DEPTH - 1; ++d) issue(first + d * step, d);
  float mu_n = 0.f, r_n = 0.f;            // the row statistics travel one step ahead in registers
  if (cact && first < rows) { mu_n = mu_i[first]; r_n = r_i[first]; }
  int it = 0;
  for (long long base = static_cast<long long>(blockIdx.x) * RPB; base < rows; base += step, ++it) {
    const long long row = base + rslot;
    const bool act = cact && row < rows;
    issue(row + (LN_DEPTH - 1) * step, (it + LN_DEPTH - 1) % LN_DEPTH);
    const float mu = mu_n, r = r_n;
    if (cact && row + step < rows) { mu_n = mu_i[row + step]; r_n = r_i[row + step]; }
    cp_async_wait<LN_DEPTH - 1>();
    const uint4* src = mine + (it % LN_DEPTH) * 3 * ROW_THREADS;
    float xh[8], dxh[8], dz[8], uh[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) xh[i] = dxh[i] = dz[i] = uh[i] = 0.f;
    if (act) {
      Raw8<bf16> xc;
      Raw8<TZ> zc;
      xc.v = src[0];
      zc.v = src[ROW_THREADS];
      float x[8];
      cvt8(xc, x);
      cvt8(zc, dz);
      if (U != nullptr) {
        Raw8<bf16> uc;
        uc.v = src[2 * ROW_THREADS];
        float u[8], a[8], b[8];
        cvt8(uc, u);
        lds8v(sp, a);
        lds8v(sp + Cs, b);
#pragma unroll
        for (int i = 0; i < 8; ++i) xh[i] = (fmaf(a[i], u[i], b[i]) + x[i] - mu) * r;
        lds8v(sp + 3 * Cs, a);
        lds8v(sp + 4 * Cs, b);
#pragma unroll
        for (int i = 0; i < 8; ++i) uh[i] = (u[i] - a[i]) * b[i];
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) xh[i] = (x[i] - mu) * r;
      }
      float w[8];
      lds8v(sp + 2 * Cs, w);
#pragma unroll
      for (int i = 0; i < 8; ++i) dxh[i] = dz[i] * w[i];
    }
    float s2[2] = {0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      s2[0] += dxh[i];
      s2[1] = fmaf(dxh[i], xh[i], s2[1]);
    }
    row_reduce<2>(s2, S, rslot, slice, red, buf);
    if (act) {
      const float m1 = s2[0] * invC, m2 = s2[1] * invC;
      float dv[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        dv[i] = r * (dxh[i] - m1 - xh[i] * m2);
        g_lw[i] = fmaf(dz[i], xh[i], g_lw[i]);
        g_lb[i] += dz[i];
        g_ga[i] = fmaf(dv[i], uh[i], g_ga[i]);
        g_be[i] += dv[i];
      }
      store8(dV + row * C + c0, dv);
    }
  }
  cp_async_wait<0>();
  __syncthreads();
  float (*acc_sm)[4][ACC_PITCH] = reinterpret_cast<float (*)[4][ACC_PITCH]>(smbuf);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    acc_sm[warp][0][lane * 8 + i] = g_lw[i];
    acc_sm[warp][1][lane * 8 + i] = g_lb[i];
    acc_sm[warp][2][lane * 8 + i] = g_ga[i];
    acc_sm[warp][3][lane * 8 + i] = g_be[i];
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < 4 * S * 256; idx += ROW_THREADS) {
    const int st = idx / (S * 256), cc = idx % (S * 256);
    const int sl = cc / 256, ci = cc % 256;
    if (cc < C) {
      float t = 0.f;
      for (int rs = 0; rs < RPB; ++rs) t += acc_sm[rs * S + sl][st][ci];
      part[(static_cast<long long>(blockIdx.x) * 4 + st) * C + cc] = t;
    }
  }
}

// partials [np][4][C] -> parameter gradients + dU coefficient vectors: dU = k1*dV + k2*U + k3   (SURVEY §8a row 10)
__global__ void __launch_bounds__(32 * RED_Y)
    bn_bwd_finalize_kernel(const float* __restrict__ part, int np, int C, double count,
                           const float* __restrict__ gamma, const float* __restrict__ bn_mean,
                           const float* __restrict__ bn_rstd, int training, int bn_layer, float* __restrict__ d_lnw,
                           float* __restrict__ d_lnb, float* __restrict__ d_gamma, float* __restrict__ d_beta,
                           float* __restrict__ d_bz, float* __restrict__ k1, float* __restrict__ k2,
                           float* __restrict__ k3) {
  __shared__ double sm[4][RED_Y][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const bool cact = c < C;
  double s[4];
  reduce_partial_rows<4>(part, np, 4LL * C, C, c, cact, s, sm);
  if (threadIdx.y != 0 || !cact) return;
  d_lnw[c] = static_cast<float>(s[0]);
  d_lnb[c] = static_cast<float>(s[1]);
  if (!bn_layer) {
    if (d_gamma) d_gamma[c] = 0.f;
    if (d_beta) d_beta[c] = 0.f;
    d_bz[c] = static_cast<float>(s[3]);  // dU = dV
    k1[c] = 1.f; k2[c] = 0.f; k3[c] = 0.f;
    return;
  }
  d_gamma[c] = static_cast<float>(s[2]);
  d_beta[c] = static_cast<float>(s[3]);
  const double g = gamma[c], rstd = bn_rstd[c], mean = bn_mean[c];
  if (training) {
    const double mdv = s[3] / count, mdvu = s[2] / count;
    k1[c] = static_cast<float>(g * rstd);
    k2[c] = static_cast<float>(-g * rstd * rstd * mdvu);
    k3[c] = static_cast<float>(-g * rstd * mdv + g * rstd * rstd * mean * mdvu);
    d_bz[c] = 0.f;  // train-mode BN cancels any per-channel shift of U: the gradient is analytically zero
  } else {
    k1[c] = static_cast<float>(g * rstd);
    k2[c] = 0.f;
    k3[c] = 0.f;
    d_bz[c] = static_cast<float>(g * rstd * s[3]);
  }
}

// dU = k1*dV + k2*U + k3 (per channel), 8 channels per thread
template <typename TA>
__global__ void bn_bwd_apply_kernel(const TA* __restrict__ dV, const TA* __restrict__ U,
                                    const float* __restrict__ k1, const float* __restrict__ k2,
                                    const float* __restrict__ k3, TA* __restrict__ dU, long long nvec, int C) {
  const int cv = C / 8;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < nvec;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c0 = static_cast<int>(i % cv) * 8;
    float a[8], b[8], c[8], dv[8], u[8], o[8];
    load8(k1 + c0, a); load8(k2 + c0, b); load8(k3 + c0, c);
    load8(dV + i * 8, dv);
    load8(U + i * 8, u);
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = fmaf(a[j], dv[j], fmaf(b[j], u[j], c[j]));
    store8(dU + i * 8, o);
  }
}

// ------------------------------------------------------------------------------------------------ reductions / casts
// out[c] = alpha * sum_i part[i*stride + c]  (fixed order)
__global__ void __launch_bounds__(32 * RED_Y)
    reduce_partials_kernel(const float* __restrict__ part, int np, long long stride, int n, float alpha,
                           float* __restrict__ out) {
  __shared__ double sm[1][RED_Y][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const bool cact = c < n;
  double s[1];
  reduce_partial_rows<1>(part, np, stride, 0, c, cact, s, sm);
  if (threadIdx.y == 0 && cact) out[c] = static_cast<float>(s[0] * alpha);
}

// three reductions in one launch (blockIdx.y selects): the bias gradients of theta / phi / g
struct Reduce3 {
  const float* part[3];
  float* out[3];
};
__global__ void __launch_bounds__(32 * RED_Y)
    reduce_partials3_kernel(const Reduce3 r, int np, long long stride, int n) {
  __shared__ double sm[1][RED_Y][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const bool cact = c < n;
  double s[1];
  reduce_partial_rows<1>(r.part[blockIdx.y], np, stride, 0, c, cact, s, sm);
  if (threadIdx.y == 0 && cact) r.out[blockIdx.y][c] = static_cast<float>(s[0]);
}

// fp32 -> bf16 (8 elements per thread)
__global__ void cast_bf16_kernel(const float* __restrict__ in, bf16* __restrict__ out, long long nvec) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < nvec;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float f[8];
    load8(in + i * 8, f);
    store8(out + i * 8, f);
  }
}

// fp32 -> three bf16 limb planes (hi, mid, lo): x = l0 + l1 + l2 to 24 mantissa bits.  out: [3][n]
__global__ void split3_kernel(const float* __restrict__ in, bf16* __restrict__ out, long long nvec, long long plane) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < nvec;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float f[8], h[8], m[8], l[8];
    load8(in + i * 8, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      h[j] = __bfloat162float(__float2bfloat16(f[j]));
      const float r1 = f[j] - h[j];
      m[j] = __bfloat162float(__float2bfloat16(r1));
      l[j] = r1 - m[j];
    }
    store8(out + i * 8, h);
    store8(out + plane + i * 8, m);
    store8(out + 2 * plane + i * 8, l);
  }
}

// per-CTA partial column sums / sums of squares of an fp32 [rows, C] matrix: part [gridDim.x][2][C]
__global__ void __launch_bounds__(256) colstats_f32_kernel(const float* __restrict__ A, float* __restrict__ part,
                                                           long long rows, int C) {
  // thread (tx = column group of 4, ty = row lane); 64 column groups x 4 row lanes per pass over 256 columns
  __shared__ float sm[2][4][256];
  for (int cbase = 0; cbase < C; cbase += 256) {
    const int c = cbase + (threadIdx.x & 63) * 4;
    const int ty = threadIdx.x >> 6;
    float s[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
    if (c < C) {
      for (long long r = static_cast<long long>(blockIdx.x) * 4 + ty; r < rows; r += static_cast<long long>(gridDim.x) * 4) {
        const float4 v = *reinterpret_cast<const float4*>(A + r * C + c);
        s[0] += v.x; s[1] += v.y; s[2] += v.z; s[3] += v.w;
        s2[0] = fmaf(v.x, v.x, s2[0]); s2[1] = fmaf(v.y, v.y, s2[1]);
        s2[2] = fmaf(v.z, v.z, s2[2]); s2[3] = fmaf(v.w, v.w, s2[3]);
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      sm[0][ty][(threadIdx.x & 63) * 4 + j] = s[j];
      sm[1][ty][(threadIdx.x & 63) * 4 + j] = s2[j];
    }
    __syncthreads();
    const int cc = cbase + threadIdx.x;
    if (cc < C) {
      const float a = sm[0][0][threadIdx.x] + sm[0][1][threadIdx.x] + sm[0][2][threadIdx.x] + sm[0][3][threadIdx.x];
      const float a2 = sm[1][0][threadIdx.x] + sm[1][1][threadIdx.x] + sm[1][2][threadIdx.x] + sm[1][3][threadIdx.x];
      part[(static_cast<long long>(blockIdx.x) * 2) * C + cc] = a;
      part[(static_cast<long long>(blockIdx.x) * 2 + 1) * C + cc] = a2;
    }
    __syncthreads();
  }
}

// fp32 concatenated weights for the F32X3 path: Wcat [3Ci, C], WcatT [C, 3Ci], bcat [3Ci]
__global__ void prep_weights_f32_kernel(const float* __restrict__ tw, const float* __restrict__ pw,
                                        const float* __restrict__ gw, const float* __restrict__ tb,
                                        const float* __restrict__ pb, const float* __restrict__ gb,
                                        float* __restrict__ wcat, float* __restrict__ wcatT, float* __restrict__ bcat,
                                        int C, int Ci) {
  const int total = 3 * Ci * C;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int r = i / C, c = i % C;
    const int which = r / Ci, rr = r % Ci;
    const float v = (which == 0 ? tw : (which == 1 ? pw : gw))[rr * C + c];
    wcat[i] = v;
    wcatT[static_cast<long long>(c) * 3 * Ci + r] = v;
    if (i < 3 * Ci) bcat[i] = ((i / Ci) == 0 ? tb : ((i / Ci) == 1 ? pb : gb))[i % Ci];
  }
}

template <typename... P>
bool aligned16(const P*... ptrs) {
  return (((reinterpret_cast<uintptr_t>(ptrs)) | ...) & 15) == 0;
}
int row_grid(long long rows, int S) {
  const int RPB = ROW_WARPS / S;
  long long blocks = (rows + RPB - 1) / RPB;
  const long long cap = 148 * 8;
  return static_cast<int>(blocks < cap ? (blocks < 1 ? 1 : blocks) : cap);
}

// ------------------------------------------------------------------------------------------------ 2-byte parameters
// blockIdx.y = tensor; 8-element vectors where both pointers are 16-byte aligned, elements otherwise.  The conversion is
// exact towards fp32 and rounds to nearest away from it (static_cast / pack2), so an fp16 overflow becomes +-inf.
template <typename TS, typename TD>
__global__ void __launch_bounds__(256) convert_params_kernel(const ParamCopy p) {
  const int k = blockIdx.y;
  const TS* __restrict__ src = static_cast<const TS*>(p.src[k]);
  TD* __restrict__ dst = static_cast<TD*>(p.dst[k]);
  if (src == nullptr || dst == nullptr) return;
  const long long n = p.n[k];
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  long long head = 0;
  if (((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0) {
    head = n / 8;
    for (long long v = t; v < head; v += stride) {
      float f[8];
      load8(src + 8 * v, f);
      store8(dst + 8 * v, f);
    }
    head *= 8;
  }
  for (long long i = head + t; i < n; i += stride) dst[i] = static_cast<TD>(static_cast<float>(src[i]));
}

}  // namespace

// ------------------------------------------------------------------------------------------------ host launchers
int convert_params(const ParamCopy& p, int src_dtype, int dst_dtype, cudaStream_t stream) {
  long long nmax = 0;
  for (int k = 0; k < NPARAMS; ++k) nmax = p.n[k] > nmax ? p.n[k] : nmax;
  long long gx = (nmax + 8 * 256 - 1) / (8 * 256);
  gx = gx < 1 ? 1 : (gx > 128 ? 128 : gx);
  const dim3 grid(static_cast<unsigned>(gx), NPARAMS);
  if (src_dtype == GLF_DTYPE_BF16 && dst_dtype == GLF_DTYPE_F32) convert_params_kernel<bf16, float><<<grid, 256, 0, stream>>>(p);
  else if (src_dtype == GLF_DTYPE_F16 && dst_dtype == GLF_DTYPE_F32) convert_params_kernel<f16, float><<<grid, 256, 0, stream>>>(p);
  else if (src_dtype == GLF_DTYPE_F32 && dst_dtype == GLF_DTYPE_BF16) convert_params_kernel<float, bf16><<<grid, 256, 0, stream>>>(p);
  else if (src_dtype == GLF_DTYPE_F32 && dst_dtype == GLF_DTYPE_F16) convert_params_kernel<float, f16><<<grid, 256, 0, stream>>>(p);
  else return set_error(GLF_ERR_INVALID, "convert_params: fp32 <-> bf16 / fp16 only");
  return check_cuda(cudaGetLastError(), "convert_params launch");
}

int transpose_cast(const void* in, void* out, int batch, int R, int S, int in_dtype, int out_dtype,
                   cudaStream_t stream) {
  if (batch <= 0 || R <= 0 || S <= 0) return set_error(GLF_ERR_INVALID, "transpose: empty");
  dim3 grid((S + 63) / 64, (R + 63) / 64, batch);
  if (grid.y > 65535 || grid.z > 65535) return set_error(GLF_ERR_INVALID, "transpose: grid too large");
  auto valid = [](int t) { return t == GLF_DTYPE_BF16 || t == GLF_DTYPE_F32 || t == GLF_DTYPE_F16; };
  if (!valid(in_dtype) || !valid(out_dtype)) return set_error(GLF_ERR_INVALID, "transpose: bad dtype");
  auto launch = [&](auto tin) {
    using TI = decltype(tin);
    const TI* src = reinterpret_cast<const TI*>(in);
    if (out_dtype == GLF_DTYPE_BF16)
      transpose_kernel<TI, bf16><<<grid, 256, 0, stream>>>(src, reinterpret_cast<bf16*>(out), R, S);
    else if (out_dtype == GLF_DTYPE_F16)
      transpose_kernel<TI, f16><<<grid, 256, 0, stream>>>(src, reinterpret_cast<f16*>(out), R, S);
    else
      transpose_kernel<TI, float><<<grid, 256, 0, stream>>>(src, reinterpret_cast<float*>(out), R, S);
  };
  if (in_dtype == GLF_DTYPE_BF16) launch(bf16{});
  else if (in_dtype == GLF_DTYPE_F16) launch(f16{});
  else launch(float{});
  return check_cuda(cudaGetLastError(), "transpose launch");
}

int prep_weights(const glf_weights* w, int C, int Ci, bf16* wcat, bf16* wcatT, float* bcat, bf16* wz, bf16* wzT,
                 cudaStream_t stream) {
  const int blocks = 4 * ((C + 31) / 32) * ((Ci + 31) / 32);      // three projections + W_z, 32 x 32 tiles
  prep_weights_kernel<<<blocks, 256, 0, stream>>>(w->theta_w, w->phi_w, w->g_w, w->theta_b, w->phi_b, w->g_b, w->wz_w,
                                                  wcat, wcatT, bcat, wz, wzT, C, Ci);
  return check_cuda(cudaGetLastError(), "prep_weights launch");
}

namespace {
// mode='gaussian': wg = bf16(g.weight) [Ci, C], bg [Ci], wgT [C, 2C + Ci] = [I | I | g.weight^T], and W_z as
// prep_weights_kernel writes it.  One element per thread (grid-stride): the transposed reads of g.weight / W_z are
// strided, which a per-call pass over C (2C + Ci) elements can afford.
__global__ void __launch_bounds__(256) prep_weights_gaussian_kernel(const float* __restrict__ gw,
                                                                     const float* __restrict__ gb,
                                                                     const float* __restrict__ wz, bf16* __restrict__ wg,
                                                                     bf16* __restrict__ wgT, float* __restrict__ bg,
                                                                     bf16* __restrict__ wzb, bf16* __restrict__ wzT,
                                                                     int C, int Ci) {
  const long long W = 2LL * C + Ci;
  const long long n_t = static_cast<long long>(C) * W, n_w = static_cast<long long>(Ci) * C;
  const long long total = n_t + 2 * n_w + Ci;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    if (i < n_t) {
      const long long c = i / W, k = i % W;
      float v;
      if (k < 2LL * C) v = (k % C) == c ? 1.f : 0.f;
      else v = gw[(k - 2LL * C) * C + c];
      wgT[i] = __float2bfloat16(v);
    } else if (i < n_t + n_w) {
      const long long j = i - n_t;                         // g.weight, row-major [Ci, C]
      wg[j] = __float2bfloat16(gw[j]);
    } else if (i < n_t + 2 * n_w) {
      const long long j = i - n_t - n_w;                   // W_z [C, Ci] and its transpose [Ci, C]
      const float v = wz[j];
      wzb[j] = __float2bfloat16(v);
      wzT[(j % Ci) * C + j / Ci] = __float2bfloat16(v);
    } else {
      const long long j = i - n_t - 2 * n_w;
      bg[j] = gb[j];
    }
  }
}
}  // namespace

int prep_weights_gaussian(const glf_weights* w, int C, int Ci, bf16* wg, bf16* wgT, float* bg, bf16* wz, bf16* wzT,
                          cudaStream_t stream) {
  const long long total = static_cast<long long>(C) * (2LL * C + Ci) + 2LL * Ci * C + Ci;
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  prep_weights_gaussian_kernel<<<static_cast<unsigned>(blocks), 256, 0, stream>>>(w->g_w, w->g_b, w->wz_w, wg, wgT, bg,
                                                                                  wz, wzT, C, Ci);
  return check_cuda(cudaGetLastError(), "prep_weights_gaussian launch");
}

// stage-1 launcher: returns the reduced table (in `scratch`) and its row count through *np
int reduce_stage1(const float* p0, const float* p1, const float* p2, int ntab, const int* np_in, int* np,
                  long long* row_stride, long long stat_stride, int NS, int C, float* scratch, cudaStream_t stream) {
  // rows of the reduced table: enough groups that each of a block's RED_Y row-threads sums ~4 partial rows, never
  // more than the scratch holds (a table of a few hundred rows needs a handful of blocks per channel slab, not 64)
  int np_max = 0;
  for (int i = 0; i < ntab; ++i) np_max = np_in[i] > np_max ? np_in[i] : np_max;
  int G = (np_max + 4 * RED_Y - 1) / (4 * RED_Y);
  G = G < 1 ? 1 : (G > REDUCE_STAGE1_ROWS ? REDUCE_STAGE1_ROWS : G);
  Stage1 t;
  const long long tab = static_cast<long long>(REDUCE_STAGE1_ROWS) * NS * C;   // table pitch in the scratch: fixed, whatever G
  t.part[0] = p0; t.part[1] = p1; t.part[2] = p2;
  t.out[0] = scratch; t.out[1] = scratch + tab; t.out[2] = scratch + 2 * tab;
  for (int i = 0; i < 3; ++i) t.np[i] = i < ntab ? np_in[i] : 0;
  dim3 grid((C + 31) / 32, G, ntab);
  if (NS == 1) reduce_stage1_kernel<1><<<grid, dim3(32, RED_Y), 0, stream>>>(t, *row_stride, stat_stride, C, G);
  else reduce_stage1_kernel<2><<<grid, dim3(32, RED_Y), 0, stream>>>(t, *row_stride, stat_stride, C, G);
  *np = G;
  *row_stride = static_cast<long long>(NS) * C;
  return check_cuda(cudaGetLastError(), "reduce_stage1 launch");
}

int bn_finalize(const float* part, int np, int C, double count, const glf_desc* d, const glf_weights* w, const float* bz,
                float* mean, float* rstd, float* a, float* b, cudaStream_t stream) {
  auto launch = [&](auto* tag) {
    using TR = std::remove_pointer_t<decltype(tag)>;
    bn_finalize_kernel<TR><<<(C + 31) / 32, dim3(32, RED_Y), 0, stream>>>(
        part, np, C, count, w->bn_w, w->bn_b, bz, d->eps_bn, d->momentum, d->training, d->bn_layer,
        reinterpret_cast<TR*>(w->bn_running_mean), reinterpret_cast<TR*>(w->bn_running_var),
        reinterpret_cast<long long*>(w->bn_num_batches_tracked), mean, rstd, a, b);
  };
  const int rdt = param_dtype(d);    // the running statistics are stored like the parameters
  if (rdt == GLF_DTYPE_BF16) launch(static_cast<bf16*>(nullptr));
  else if (rdt == GLF_DTYPE_F16) launch(static_cast<f16*>(nullptr));
  else launch(static_cast<float*>(nullptr));
  return check_cuda(cudaGetLastError(), "bn_finalize launch");
}

int bn_res_ln_fwd(const void* U_, const void* X_, int act_dtype, const float* a, const float* b, const float* lw,
                  const float* lb, void* Z, int z_dtype, float* mu, float* r, long long rows, int C, float eps,
                  int accumulate, cudaStream_t stream) {
  if (C % 8 != 0 || C > 2048) return set_error(GLF_ERR_INVALID, "LayerNorm kernel needs C %% 8 == 0 and C <= 2048");
  if (z_dtype == GLF_DTYPE_F16 && act_dtype != GLF_DTYPE_BF16)
    return set_error(GLF_ERR_INVALID, "LayerNorm kernel: an fp16 Z needs bf16 activations");
  const bool z16 = z_dtype == GLF_DTYPE_BF16 || z_dtype == GLF_DTYPE_F16;    // bf16 or fp16 Z: the fast paths
  if (act_dtype == GLF_DTYPE_BF16 && z16 && U_ != nullptr && ln_tma_supported(C) &&
      aligned16(U_, X_, Z, a, b, lw, lb)) {
    const bf16* Ua[1] = {(const bf16*)U_};
    const bf16* Xa[1] = {(const bf16*)X_};
    const float *aa[1] = {a}, *ba[1] = {b}, *lwa[1] = {lw}, *lba[1] = {lb};
    float *mua[1] = {mu}, *ra[1] = {r};
    return ln_fwd_tma(1, Ua, Xa, aa, ba, lwa, lba, mua, ra, Z, rows, C, eps, accumulate, stream, nullptr, z_dtype);
  }
  int S = (C + 255) / 256;
  while (ROW_WARPS % S != 0) ++S;
  const int grid = row_grid(rows, S);
  if (act_dtype == GLF_DTYPE_BF16) {
    const bf16* U = (const bf16*)U_; const bf16* X = (const bf16*)X_;
    if (S > 1 && z16 && aligned16(U_ != nullptr ? U_ : X_, X_, Z)) {
      const size_t ring = LN_DEPTH * 3 * ROW_THREADS * sizeof(uint4);       // 48 KB
      const void* kern = z_dtype == GLF_DTYPE_F16 ? reinterpret_cast<const void*>(bn_res_ln_fwd_ring_kernel<f16>)
                                                  : reinterpret_cast<const void*>(bn_res_ln_fwd_ring_kernel<bf16>);
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(ring));
      if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(ln fwd ring)");
      if (z_dtype == GLF_DTYPE_F16)
        bn_res_ln_fwd_ring_kernel<f16><<<grid, ROW_THREADS, ring, stream>>>(U, X, a, b, lw, lb, (f16*)Z, mu, r, rows, C, S, eps, accumulate);
      else
        bn_res_ln_fwd_ring_kernel<bf16><<<grid, ROW_THREADS, ring, stream>>>(U, X, a, b, lw, lb, (bf16*)Z, mu, r, rows, C, S, eps, accumulate);
    } else if (z_dtype == GLF_DTYPE_BF16)
      bn_res_ln_fwd_kernel<bf16, bf16><<<grid, ROW_THREADS, 0, stream>>>(U, X, a, b, lw, lb, (bf16*)Z, mu, r, rows, C, S, eps, accumulate);
    else if (z_dtype == GLF_DTYPE_F16)
      bn_res_ln_fwd_kernel<f16, bf16><<<grid, ROW_THREADS, 0, stream>>>(U, X, a, b, lw, lb, (f16*)Z, mu, r, rows, C, S, eps, accumulate);
    else
      bn_res_ln_fwd_kernel<float, bf16><<<grid, ROW_THREADS, 0, stream>>>(U, X, a, b, lw, lb, (float*)Z, mu, r, rows, C, S, eps, accumulate);
  } else {
    const float* U = (const float*)U_; const float* X = (const float*)X_;
    if (z_dtype == GLF_DTYPE_BF16)
      bn_res_ln_fwd_kernel<bf16, float><<<grid, ROW_THREADS, 0, stream>>>(U, X, a, b, lw, lb, (bf16*)Z, mu, r, rows, C, S, eps, accumulate);
    else
      bn_res_ln_fwd_kernel<float, float><<<grid, ROW_THREADS, 0, stream>>>(U, X, a, b, lw, lb, (float*)Z, mu, r, rows, C, S, eps, accumulate);
  }
  return check_cuda(cudaGetLastError(), "bn_res_ln_fwd launch");
}

// fused pair forward for wide rows (256 < C <= 2048, bf16): see ln_pair_fwd_ring_kernel
bool ln_pair_wide_supported(int C) { return C > 256 && C <= 2048 && C % 8 == 0; }

int ln_pair_fwd_wide(const bf16* const* U, const bf16* const* X, const float* const* a, const float* const* b,
                     const float* const* lw, const float* const* lb, float* const* mu, float* const* r, void* Z,
                     long long rows, int C, float eps, int accumulate, cudaStream_t stream, void* Z0, int z_dtype) {
  if (!ln_pair_wide_supported(C)) return set_error(GLF_ERR_UNSUPPORTED, "ln_pair_fwd_wide: 256 < C <= 2048 expected");
  if (z_dtype != GLF_DTYPE_BF16 && z_dtype != GLF_DTYPE_F16) return set_error(GLF_ERR_INVALID, "ln_pair_fwd_wide: Z must be bf16 or fp16");
  if (Z0 != nullptr && accumulate) return set_error(GLF_ERR_INVALID, "ln_pair_fwd_wide: parts with accumulate");
  int S = (C + 255) / 256;
  while (ROW_WARPS % S != 0) ++S;
  LnPairWide p;
  for (int m = 0; m < 2; ++m) {
    p.U[m] = U[m]; p.X[m] = X[m]; p.a[m] = a[m]; p.b[m] = b[m]; p.lw[m] = lw[m]; p.lb[m] = lb[m];
    p.mu[m] = mu[m]; p.r[m] = r[m];
    if (U[m] == nullptr || !aligned16(U[m], X[m])) return set_error(GLF_ERR_INVALID, "ln_pair_fwd_wide: operands must be 16-byte aligned");
  }
  if (!aligned16(Z, Z0 != nullptr ? Z0 : Z)) return set_error(GLF_ERR_INVALID, "ln_pair_fwd_wide: outputs must be 16-byte aligned");
  p.Z = Z; p.Z0 = Z0; p.rows = rows; p.C = C; p.S = S; p.accumulate = accumulate; p.eps = eps;
  const int grid = row_grid(rows, S);
  const size_t ring = LN_DEPTH * 5 * ROW_THREADS * sizeof(uint4);       // 80 KB
  const bool h = z_dtype == GLF_DTYPE_F16;
  void (*kern)(const LnPairWide) =
      Z0 != nullptr ? (h ? ln_pair_fwd_ring_kernel<true, f16> : ln_pair_fwd_ring_kernel<true, bf16>)
                    : (h ? ln_pair_fwd_ring_kernel<false, f16> : ln_pair_fwd_ring_kernel<false, bf16>);
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(ring));
  if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(ln pair wide)");
  kern<<<grid, ROW_THREADS, ring, stream>>>(p);
  return check_cuda(cudaGetLastError(), "ln_pair_fwd_wide launch");
}

int bn_res_ln_bwd_blocks(long long rows, int C) {
  int S = (C + 255) / 256;
  while (ROW_WARPS % S != 0) ++S;
  const int g = row_grid(rows, S);
  return g < 148 * 2 ? g : 148 * 2;
}

int bn_res_ln_bwd(const void* dZ, int dz_dtype, const void* U_, const void* X_, int act_dtype, const float* a,
                  const float* b, const float* mean, const float* rstd, const float* lw, const float* mu,
                  const float* r, void* dV_, float* part, long long rows, int C, int* nblocks, cudaStream_t stream) {
  if (C % 8 != 0 || C > 2048) return set_error(GLF_ERR_INVALID, "LayerNorm kernel needs C %% 8 == 0 and C <= 2048");
  if (dz_dtype == GLF_DTYPE_F16 && act_dtype != GLF_DTYPE_BF16)
    return set_error(GLF_ERR_INVALID, "LayerNorm backward: an fp16 dZ needs bf16 activations");
  const bool dz16 = dz_dtype == GLF_DTYPE_BF16 || dz_dtype == GLF_DTYPE_F16;  // bf16 or fp16 dZ: the fast paths
  if (act_dtype == GLF_DTYPE_BF16 && dz16 && U_ != nullptr && ln_tma_supported(C) &&
      aligned16(dZ, U_, X_, dV_, a, b, lw, mu, r)) {
    const bf16* Ua[1] = {(const bf16*)U_};
    const bf16* Xa[1] = {(const bf16*)X_};
    const float *aa[1] = {a}, *ba[1] = {b}, *lwa[1] = {lw}, *mna[1] = {mean}, *rsa[1] = {rstd}, *mua[1] = {mu},
                *ra[1] = {r};
    bf16* dVa[1] = {(bf16*)dV_};
    float* pa[1] = {part};
    return ln_bwd_tma(1, dZ, Ua, Xa, aa, ba, lwa, mna, rsa, mua, ra, dVa, pa, rows, C, nblocks, stream, 0, nullptr, nullptr,
                      0, dz_dtype);
  }
  int S = (C + 255) / 256;
  while (ROW_WARPS % S != 0) ++S;
  const int grid = bn_res_ln_bwd_blocks(rows, C);
  if (nblocks) *nblocks = grid;
  if (act_dtype == GLF_DTYPE_BF16) {
    const bf16* U = (const bf16*)U_; const bf16* X = (const bf16*)X_; bf16* dV = (bf16*)dV_;
    if (S > 1 && dz16 && aligned16(U_ != nullptr ? U_ : X_, X_, dZ, dV_)) {
      const size_t ring = LN_DEPTH * 3 * ROW_THREADS * sizeof(uint4);
      const void* kern = dz_dtype == GLF_DTYPE_F16 ? reinterpret_cast<const void*>(bn_res_ln_bwd_ring_kernel<f16>)
                                                   : reinterpret_cast<const void*>(bn_res_ln_bwd_ring_kernel<bf16>);
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(ring));
      if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(ln bwd ring)");
      if (dz_dtype == GLF_DTYPE_F16)
        bn_res_ln_bwd_ring_kernel<f16><<<grid, ROW_THREADS, ring, stream>>>((const f16*)dZ, U, X, a, b, mean, rstd, lw, mu, r, dV, part, rows, C, S);
      else
        bn_res_ln_bwd_ring_kernel<bf16><<<grid, ROW_THREADS, ring, stream>>>((const bf16*)dZ, U, X, a, b, mean, rstd, lw, mu, r, dV, part, rows, C, S);
    } else if (dz_dtype == GLF_DTYPE_BF16)
      bn_res_ln_bwd_kernel<bf16, bf16><<<grid, ROW_THREADS, 0, stream>>>((const bf16*)dZ, U, X, a, b, mean, rstd, lw, mu, r, dV, part, rows, C, S);
    else if (dz_dtype == GLF_DTYPE_F16)
      bn_res_ln_bwd_kernel<f16, bf16><<<grid, ROW_THREADS, 0, stream>>>((const f16*)dZ, U, X, a, b, mean, rstd, lw, mu, r, dV, part, rows, C, S);
    else
      bn_res_ln_bwd_kernel<float, bf16><<<grid, ROW_THREADS, 0, stream>>>((const float*)dZ, U, X, a, b, mean, rstd, lw, mu, r, dV, part, rows, C, S);
  } else {
    const float* U = (const float*)U_; const float* X = (const float*)X_; float* dV = (float*)dV_;
    if (dz_dtype == GLF_DTYPE_BF16)
      bn_res_ln_bwd_kernel<bf16, float><<<grid, ROW_THREADS, 0, stream>>>((const bf16*)dZ, U, X, a, b, mean, rstd, lw, mu, r, dV, part, rows, C, S);
    else
      bn_res_ln_bwd_kernel<float, float><<<grid, ROW_THREADS, 0, stream>>>((const float*)dZ, U, X, a, b, mean, rstd, lw, mu, r, dV, part, rows, C, S);
  }
  return check_cuda(cudaGetLastError(), "bn_res_ln_bwd launch");
}

int bn_bwd_finalize(const float* part, int np, int C, double count, const glf_desc* d, const glf_weights* w,
                    const float* mean, const float* rstd, const glf_grads* g, float* k1, float* k2, float* k3,
                    cudaStream_t stream) {
  bn_bwd_finalize_kernel<<<(C + 31) / 32, dim3(32, RED_Y), 0, stream>>>(part, np, C, count, w->bn_w, mean, rstd, d->training,
                                                              d->bn_layer, g->ln_w, g->ln_b, g->bn_w, g->bn_b, g->wz_b,
                                                              k1, k2, k3);
  return check_cuda(cudaGetLastError(), "bn_bwd_finalize launch");
}

int bn_bwd_apply(const void* dV, const void* U, int act_dtype, const float* k1, const float* k2, const float* k3,
                 void* dU, long long rows, int C, cudaStream_t stream) {
  const long long nvec = rows * C / 8;
  long long blocks = (nvec + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (act_dtype == GLF_DTYPE_BF16)
    bn_bwd_apply_kernel<bf16><<<static_cast<int>(blocks), 256, 0, stream>>>((const bf16*)dV, (const bf16*)U, k1, k2, k3, (bf16*)dU, nvec, C);
  else
    bn_bwd_apply_kernel<float><<<static_cast<int>(blocks), 256, 0, stream>>>((const float*)dV, (const float*)U, k1, k2, k3, (float*)dU, nvec, C);
  return check_cuda(cudaGetLastError(), "bn_bwd_apply launch");
}

int reduce_partials(const float* part, int np, long long stride, int n, float alpha, float* out, cudaStream_t stream) {
  reduce_partials_kernel<<<(n + 31) / 32, dim3(32, RED_Y), 0, stream>>>(part, np, stride, n, alpha, out);
  return check_cuda(cudaGetLastError(), "reduce_partials launch");
}

int reduce_partials3(const float* p0, const float* p1, const float* p2, int np, long long stride, int n, float* o0,
                     float* o1, float* o2, cudaStream_t stream) {
  Reduce3 r;
  r.part[0] = p0; r.part[1] = p1; r.part[2] = p2;
  r.out[0] = o0; r.out[1] = o1; r.out[2] = o2;
  reduce_partials3_kernel<<<dim3((n + 31) / 32, 3), dim3(32, RED_Y), 0, stream>>>(r, np, stride, n);
  return check_cuda(cudaGetLastError(), "reduce_partials3 launch");
}

int split3(const float* in, bf16* out, long long n, cudaStream_t stream) {
  if (n % 8 != 0) return set_error(GLF_ERR_INVALID, "split3: n %% 8 != 0");
  const long long nvec = n / 8;
  long long blocks = (nvec + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  split3_kernel<<<static_cast<int>(blocks < 1 ? 1 : blocks), 256, 0, stream>>>(in, out, nvec, n);
  return check_cuda(cudaGetLastError(), "split3 launch");
}

int colstats_f32_blocks(long long rows) {
  long long b = (rows + 3) / 4;
  return static_cast<int>(b < 1 ? 1 : (b > 148 * 4 ? 148 * 4 : b));
}
int colstats_f32(const float* A, float* part, long long rows, int C, cudaStream_t stream) {
  if (C % 4 != 0) return set_error(GLF_ERR_INVALID, "colstats_f32: C %% 4 != 0");
  colstats_f32_kernel<<<colstats_f32_blocks(rows), 256, 0, stream>>>(A, part, rows, C);
  return check_cuda(cudaGetLastError(), "colstats_f32 launch");
}

int prep_weights_f32(const glf_weights* w, int C, int Ci, float* wcat, float* wcatT, float* bcat, cudaStream_t stream) {
  const int total = 3 * Ci * C;
  int blocks = (total + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  prep_weights_f32_kernel<<<blocks, 256, 0, stream>>>(w->theta_w, w->phi_w, w->g_w, w->theta_b, w->phi_b, w->g_b, wcat,
                                                      wcatT, bcat, C, Ci);
  return check_cuda(cudaGetLastError(), "prep_weights_f32 launch");
}

int cast_bf16(const float* in, bf16* out, long long n, cudaStream_t stream) {
  if (n % 8 != 0) return set_error(GLF_ERR_INVALID, "cast_bf16: n %% 8 != 0");
  const long long nvec = n / 8;
  long long blocks = (nvec + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  cast_bf16_kernel<<<static_cast<int>(blocks < 1 ? 1 : blocks), 256, 0, stream>>>(in, out, nvec);
  return check_cuda(cudaGetLastError(), "cast_bf16 launch");
}

}  // namespace glf
