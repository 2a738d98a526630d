// glf_wgrad.cu — the four weight-gradient sums over the sequences of the Gram form of mode='dot' (autograd of
// R/models/ours.py:866-908 in the reassociated form; oracle/tpavi_oracle.py: tpavi_dot_gram_form), C = 256, C' = 128:
//
//     dW~theta = sum_b W'_b^T dQ~_b        dWz     = sum_b dW'_b M_b
//     dW~g     = sum_b (dM_b / N)^T T~_b   dW~phi  = sum_b dT~_b S~_b
//
// As batched tile GEMMs with fp32 red.add over the batch these were four launches of 16 - 19 us each, bound by 128-fold
// atomic contention in L2 (profiles/r02_v1_launches_warm.csv).  Here they are ONE launch of K-concatenated products: the
// sum over the sequences is the K loop.  Every sequence contributes `slabs` 64-deep K slabs to a product; the slabs of
// all four products are dealt to the CTAs in proportion to their bytes (theta 4, z 2, g 2, phi 4 per sequence), each CTA
// streams its contiguous slab range once through a 4-stage TMA ring (48 KB per slab: full-width operands, nothing is
// re-read), accumulates in TMEM and writes ONE fp32 partial; wgrad_reduce_kernel then sums the partials of a product in
// a fixed order (deterministic gradients, no atomics) straight into the caller's gradient tensors.
// The homogeneous column of the augmented matrices (the bias gradients) and the rank-1 term dt s^T of dWphi are formed
// in fp32 by the SIMT warps from the staged tiles.
#include <cstdio>
#include <cstdlib>

#include "glf_internal.h"
#include "glf_ptx.cuh"

namespace glf {

namespace {

constexpr int CC = 256, CI = 128, CA = 264;
constexpr int WG_THREADS = 64 + 256;           // warp 0 TMA, warp 1 MMA, warps 2..9 SIMT / epilogue
constexpr int WG_STAGES = 4;
constexpr uint32_t WG_STAGE = 49152;           // one K slab of both operands
constexpr uint32_t WG_SMEM = WG_STAGES * WG_STAGE + 4096 + 1024;
constexpr int WG_PART = 128 * 256 + 256;       // floats per partial: the matrix + the bias vector (padded)

// Debug aid (GLF_WGRAD_TRACE=1): SM clock at a few points of selected CTAs (one per product), printed by the host.
__device__ long long g_wgrad_trace[4][8];
#define WG_TRACE(i)                                                                              \
  do {                                                                                           \
    if (p.trace && j == 0) g_wgrad_trace[prod][i] = clock64();                                   \
  } while (0)

struct WgradParams {
  int B, N, trace;
  int cta0[5];            // first CTA of product p (theta, z, g, phi); cta0[4] = number of CTAs
  const float *dcv, *tv, *dtv, *sfv;   // dc [B][C], t [B][C'], dt [B][C'], s [B][C]
  float* part;            // [n_cta][WG_PART]
};

// element (row, col) of a [R][64] SWIZZLE_128B tile
__device__ __forceinline__ float tile64(const uint8_t* tile, int row, int col) {
  return __bfloat162float(*reinterpret_cast<const bf16*>(
      tile + row * 128 + ((((col >> 3) ^ (row & 7))) << 4) + (col & 7) * 2));
}

__global__ void __launch_bounds__(WG_THREADS, 1)
    wgrad_kernel(const __grid_constant__ CUtensorMap tmWp, const __grid_constant__ CUtensorMap tmdQ,
                 const __grid_constant__ CUtensorMap tmdWp, const __grid_constant__ CUtensorMap tmM,
                 const __grid_constant__ CUtensorMap tmdM, const __grid_constant__ CUtensorMap tmT,
                 const __grid_constant__ CUtensorMap tmdT, const __grid_constant__ CUtensorMap tmS,
                 const WgradParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sgen = smem_raw + (sbase - smem_u32(smem_raw));
  float* v_bias = reinterpret_cast<float*>(sgen + WG_STAGES * WG_STAGE);   // [256] bias-gradient accumulator
  uint64_t* bars = reinterpret_cast<uint64_t*>(sgen + WG_STAGES * WG_STAGE + 2048);
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(sgen + WG_STAGES * WG_STAGE + 2048 + 128);
  auto full = [&](int s) { return smem_u32(&bars[s]); };
  auto empty = [&](int s) { return smem_u32(&bars[WG_STAGES + s]); };
  const uint32_t acc_bar = smem_u32(&bars[2 * WG_STAGES]);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // product and slab range of this CTA
  int prod = 0;
  while (prod < 3 && static_cast<int>(blockIdx.x) >= p.cta0[prod + 1]) ++prod;
  const int ncta = p.cta0[prod + 1] - p.cta0[prod], j = blockIdx.x - p.cta0[prod];
  const int spq = (prod == 0 || prod == 3) ? 4 : 2;               // slabs per sequence
  const long long total = static_cast<long long>(spq) * p.B;
  const int sl0 = static_cast<int>(total * j / ncta), sl1 = static_cast<int>(total * (j + 1) / ncta);
  const int nsl = sl1 - sl0;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmWp); tma_prefetch_desc(&tmdQ); tma_prefetch_desc(&tmdWp); tma_prefetch_desc(&tmM);
    tma_prefetch_desc(&tmdM); tma_prefetch_desc(&tmT); tma_prefetch_desc(&tmdT); tma_prefetch_desc(&tmS);
    for (int s = 0; s < WG_STAGES; ++s) {
      mbar_init(full(s), 1);
      mbar_init(empty(s), 1 + 8);
    }
    mbar_init(acc_bar, 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(tmem_holder), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_holder;
  if (threadIdx.x == 0) WG_TRACE(0);

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int it = 0; it < nsl; ++it) {
        const int sl = sl0 + it, b = sl / spq, k = sl - b * spq;
        const uint32_t fb = full(stage), sa = sbase + stage * WG_STAGE;
        mbar_wait(empty(stage), phase ^ 1u);
        mbar_expect_tx(fb, WG_STAGE);
        if (prod == 0) {          // A = W'_b rows 64k.. [64][128] ; B = dQ_b rows 64k.. [64][256]
          for (int t = 0; t < 2; ++t) tma_load_4d(&tmWp, fb, sa + t * 8192, 64 * t, 64 * k, b, 0);
          for (int t = 0; t < 4; ++t) tma_load_4d(&tmdQ, fb, sa + 16384 + t * 8192, 64 * t, 64 * k, b, 0);
        } else if (prod == 1) {   // A = dW'_b columns 64k.. [256][64] ; B = M_b rows 64k.. [64][128]
          for (int h = 0; h < 2; ++h) tma_load_4d(&tmdWp, fb, sa + h * 16384, 64 * k, 128 * h, b, 0);
          for (int t = 0; t < 2; ++t) tma_load_4d(&tmM, fb, sa + 32768 + t * 8192, 64 * t, 64 * k, b, 0);
        } else if (prod == 2) {   // A = (dM/N)_b rows 64k.. [64][128] ; B = T_b rows 64k.. [64][256]
          for (int t = 0; t < 2; ++t) tma_load_4d(&tmdM, fb, sa + t * 8192, 64 * t, 64 * k, b, 0);
          for (int t = 0; t < 4; ++t) tma_load_4d(&tmT, fb, sa + 16384 + t * 8192, 64 * t, 64 * k, b, 0);
        } else {                  // A = dT_b columns 64k.. [128][64] ; B = S_b columns 64k.. [256][64]
          tma_load_4d(&tmdT, fb, sa, 64 * k, 0, b, 0);
          for (int h = 0; h < 2; ++h) tma_load_4d(&tmS, fb, sa + 16384 + h * 16384, 64 * k, 128 * h, b, 0);
        }
        if (++stage == WG_STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int it = 0; it < nsl; ++it) {
        mbar_wait(full(stage), phase);
        tc_fence_after();
        const uint32_t sa = sbase + stage * WG_STAGE;
        const uint32_t accf = it > 0 ? 1u : 0u;
#pragma unroll
        for (int k16 = 0; k16 < 4; ++k16) {
          const uint32_t acc = (accf | (k16 > 0 ? 1u : 0u));
          if (prod == 0 || prod == 2) {
            umma_f16(tmem, make_sdesc(sa + k16 * 2048, 8192, 1024), make_sdesc(sa + 16384 + k16 * 2048, 8192, 1024),
                     make_idesc_bf16(128, 256, true, true), acc);
          } else if (prod == 1) {
            const uint64_t bd = make_sdesc(sa + 32768 + k16 * 2048, 8192, 1024);
            for (int h = 0; h < 2; ++h)
              umma_f16(tmem + h * 128, make_sdesc(sa + h * 16384 + k16 * 32, 16, 1024), bd,
                       make_idesc_bf16(128, 128, false, true), acc);
          } else {
            umma_f16(tmem, make_sdesc(sa + k16 * 32, 16, 1024), make_sdesc(sa + 16384 + k16 * 32, 16, 1024),
                     make_idesc_bf16(128, 256, false, false), acc);
          }
        }
        umma_commit(empty(stage));
        if (++stage == WG_STAGES) { stage = 0; phase ^= 1u; }
      }
      umma_commit(acc_bar);
      WG_TRACE(1);
    }
  } else {
    // ------------------------------------------------------------------------------------------ SIMT warps
    const int tid = threadIdx.x - 64;          // 0..255
    // bias gradients from the staged tiles: theta: sum_r W'[r,i] dc[r]; g: sum_i (dM/N)[i,j] t[i];
    // phi: sum_k dT[i,k] s[k] (+ N dt[i] once per sequence).  Thread pairs split the 64 slab rows / columns.
    float bacc = 0.f;
    float cacc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // products theta / g: 8 columns of this thread's chunk
    {
      int stage = 0;
      uint32_t phase = 0;
      const int i = tid & 127, half = tid >> 7;
      const int cc = tid & 15, rg = tid >> 4;                    // theta / g: column chunk (of 16), row group (of 16)
      for (int it = 0; it < nsl; ++it) {
        const int sl = sl0 + it, b = sl / spq, k = sl - b * spq;
        mbar_wait(full(stage), phase);
        const uint8_t* sa = sgen + stage * WG_STAGE;
        if (prod == 0 || prod == 2) {
          const float* vec = prod == 0 ? p.dcv + static_cast<long long>(b) * CC + 64 * k
                                       : p.tv + static_cast<long long>(b) * CI + 64 * k;
          const uint8_t* tile = sa + (cc >> 3) * 8192;     // A tile ([64 rows][64 columns]) holding this column chunk
#pragma unroll
          for (int r = rg * 4; r < rg * 4 + 4; ++r) {
            const uint4 qv = *reinterpret_cast<const uint4*>(tile + r * 128 + (((cc & 7) ^ (r & 7)) << 4));
            const uint32_t* q32 = reinterpret_cast<const uint32_t*>(&qv);
            const float wv = vec[r];
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const float2 x = unpack_bf16(q32[t]);
              cacc[2 * t] = fmaf(x.x, wv, cacc[2 * t]);
              cacc[2 * t + 1] = fmaf(x.y, wv, cacc[2 * t + 1]);
            }
          }
        } else if (prod == 3) {
          const float* vec = p.sfv + static_cast<long long>(b) * CC + 64 * k;
#pragma unroll
          for (int ch = half * 4; ch < half * 4 + 4; ++ch) {
            const uint4 qv = *reinterpret_cast<const uint4*>(sa + i * 128 + ((ch ^ (i & 7)) << 4));
            const uint32_t* q32 = reinterpret_cast<const uint32_t*>(&qv);
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const float2 x = unpack_bf16(q32[t]);
              bacc = fmaf(x.x, vec[ch * 8 + 2 * t], fmaf(x.y, vec[ch * 8 + 2 * t + 1], bacc));
            }
          }
          if (k == 0 && half == 0) bacc = fmaf(static_cast<float>(p.N), p.dtv[static_cast<long long>(b) * CI + i], bacc);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty(stage));
        if (++stage == WG_STAGES) { stage = 0; phase ^= 1u; }
      }
      if (tid == 0) WG_TRACE(2);
      if (prod == 1 || prod == 3) {
        if (half == 1) v_bias[i] = bacc;
        named_bar_sync(1, 256);
        if (half == 0) v_bias[i] += bacc;
        named_bar_sync(1, 256);
      }
    }
    // ---- epilogue: fp32 partial of this CTA.  Layout [256 rows][128] for dWz, [128 rows][256] otherwise.
    const int w = warp - 2, q = warp & 3, hf = w >> 2;
    float* out = p.part + static_cast<long long>(blockIdx.x) * WG_PART;
    mbar_wait(acc_bar, 0);
    tc_fence_after();
    if (tid == 0) WG_TRACE(3);
    const int cc = tid & 15;
    if (prod == 0 || prod == 2) {    // (after the accumulator wait: the MMAs no longer read the ring)
      // 16 row groups hold partial sums of the same column chunk: lanes l and l ^ 16 first, then the 8 warps
      float* xs = reinterpret_cast<float*>(sgen);     // the ring is idle now: [8 warps][128 columns]
#pragma unroll
      for (int t = 0; t < 8; ++t) cacc[t] += __shfl_xor_sync(0xffffffffu, cacc[t], 16);
      named_bar_sync(1, 256);                          // (every warp has left the ring's last stage)
      if (lane < 16) {
#pragma unroll
        for (int t = 0; t < 8; ++t) xs[(warp - 2) * 128 + cc * 8 + t] = cacc[t];
      }
      named_bar_sync(1, 256);
      if (tid < 128) {
        float a = 0.f;
#pragma unroll
        for (int wv = 0; wv < 8; ++wv) a += xs[wv * 128 + tid];
        v_bias[tid] = a;
      }
      named_bar_sync(1, 256);
    }

    const uint32_t tlane = tmem + (static_cast<uint32_t>(q * 32) << 16);
    // the accumulator goes through the (idle) ring as fp32 rows with a padded pitch, then out with coalesced 16-byte
    // stores: thread-per-row stores straight from registers touched 32 lines per instruction
    constexpr uint32_t PITCH = 1040;                    // bytes per staged row of 256 floats (+ 4 floats: bank spread)
    uint8_t* stg = sgen + 4096;                          // (the first 4 KB held the bias exchange above)
    const int nrow = prod == 1 ? 256 : 128, ncol = prod == 1 ? 128 : 256;
    const int bs0 = (sl0 + spq - 1) / spq, bs1 = (sl1 + spq - 1) / spq;   // sequences whose slab 0 lies in [sl0, sl1)
    for (int pass = 0; pass < (prod == 1 ? 2 : 1); ++pass) {             // dWz: two 128-row halves, one at a time
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        const int srow = q * 32 + lane;
        int col0;
        uint32_t taddr;
        if (prod == 1) {
          if (hf != pass) break;                         // (warps of the other half idle in this pass)
          col0 = c * 32;
          taddr = tlane + pass * 128 + col0;
        } else {
          col0 = hf * 128 + c * 32;
          taddr = tlane + col0;
        }
        uint32_t v[32];
        tmem_ld_32x32(taddr, v);
        tmem_ld_wait();
        float f[32];
#pragma unroll
        for (int t = 0; t < 32; ++t) f[t] = __uint_as_float(v[t]);
        if (prod == 3) {       // + sum over the sequences that START in this CTA's range of dt_b[row] s_b[n]
          for (int b = bs0; b < bs1; ++b) {
            const float d = p.dtv[static_cast<long long>(b) * CI + srow];
            const float4* sv = reinterpret_cast<const float4*>(p.sfv + static_cast<long long>(b) * CC + col0);
#pragma unroll
            for (int t = 0; t < 8; ++t) {
              const float4 s4 = sv[t];
              f[4 * t] = fmaf(d, s4.x, f[4 * t]);
              f[4 * t + 1] = fmaf(d, s4.y, f[4 * t + 1]);
              f[4 * t + 2] = fmaf(d, s4.z, f[4 * t + 2]);
              f[4 * t + 3] = fmaf(d, s4.w, f[4 * t + 3]);
            }
          }
        }
        float4* dst = reinterpret_cast<float4*>(stg + srow * PITCH + col0 * 4);
#pragma unroll
        for (int t = 0; t < 8; ++t) dst[t] = make_float4(f[4 * t], f[4 * t + 1], f[4 * t + 2], f[4 * t + 3]);
      }
      named_bar_sync(1, 256);
      // 128 staged rows x ncol floats -> global rows [pass * 128, +128) of the partial
      const int v4_per_row = ncol / 4;
      float* obase = out + static_cast<long long>(pass) * 128 * ncol;
      for (int idx = tid; idx < 128 * v4_per_row; idx += 256) {
        const int r_ = idx / v4_per_row, c4 = idx - r_ * v4_per_row;
        *reinterpret_cast<float4*>(obase + static_cast<long long>(r_) * ncol + c4 * 4) =
            *reinterpret_cast<const float4*>(stg + r_ * PITCH + c4 * 16);
      }
      named_bar_sync(1, 256);
    }
    (void)nrow;
    if (tid < 128) out[128 * 256 + tid] = (prod == 1) ? 0.f : v_bias[tid];
    if (tid == 0) WG_TRACE(4);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

// Fixed-order sum of the partials of each product into the caller's gradients.
//   theta_w, phi_w, g_w [C'][C] ; theta_b, phi_b, g_b [C'] ; wz_w [C][C']
__global__ void wgrad_reduce_kernel(const float* __restrict__ part, int c0, int c1, int c2, int c3, int c4,
                                    float* __restrict__ tw, float* __restrict__ tb, float* __restrict__ zw,
                                    float* __restrict__ gw, float* __restrict__ gb, float* __restrict__ pw,
                                    float* __restrict__ pb) {
  const int per = 128 * 256 + 128;             // matrix + bias entries handled per product
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 4 * per) return;
  const int prod = idx / per, e = idx - prod * per;
  const int a = prod == 0 ? c0 : (prod == 1 ? c1 : (prod == 2 ? c2 : c3));
  const int z = prod == 0 ? c1 : (prod == 1 ? c2 : (prod == 2 ? c3 : c4));
  // four independent chains, combined in a fixed order (the partials are read with memory-level parallelism)
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  int c = a;
  for (; c + 4 <= z; c += 4) {
    a0 += part[static_cast<long long>(c) * WG_PART + e];
    a1 += part[static_cast<long long>(c + 1) * WG_PART + e];
    a2 += part[static_cast<long long>(c + 2) * WG_PART + e];
    a3 += part[static_cast<long long>(c + 3) * WG_PART + e];
  }
  for (; c < z; ++c) a0 += part[static_cast<long long>(c) * WG_PART + e];
  const float acc = (a0 + a1) + (a2 + a3);
  float* W = prod == 0 ? tw : (prod == 1 ? zw : (prod == 2 ? gw : pw));
  float* bb = prod == 0 ? tb : (prod == 1 ? nullptr : (prod == 2 ? gb : pb));
  if (e < 128 * 256) W[e] = acc;               // both layouts are the row-major layout of the gradient tensor
  else if (bb != nullptr) bb[e - 128 * 256] = acc;
}

}  // namespace

size_t gram_wgrad_scratch_floats() { return static_cast<size_t>(160) * WG_PART; }

int gram_wgrad(const bf16* Wp, const bf16* dQa, const bf16* dWp, const bf16* Mb, const bf16* dMn, const bf16* T,
               const bf16* dT, const bf16* Sa, const float* dcv, const float* tv, const float* dtv, const float* sfv,
               float* part, const glf_grads* g, int B, int N, cudaStream_t stream) {
  CUtensorMap tmWp, tmdQ, tmdWp, tmM, tmdM, tmT, tmdT, tmS;
  GLF_TRY(make_tmap_bf16(&tmWp, Wp, CI, CC, B, CI, static_cast<long long>(CC) * CI, 64));
  GLF_TRY(make_tmap_bf16(&tmdQ, dQa, CC, CC, B, CA, static_cast<long long>(CC) * CA, 64));
  GLF_TRY(make_tmap_bf16(&tmdWp, dWp, CI, CC, B, CI, static_cast<long long>(CC) * CI, 128));
  GLF_TRY(make_tmap_bf16(&tmM, Mb, CI, CI, B, CI, static_cast<long long>(CI) * CI, 64));
  GLF_TRY(make_tmap_bf16(&tmdM, dMn, CI, CI, B, CI, static_cast<long long>(CI) * CI, 64));
  GLF_TRY(make_tmap_bf16(&tmT, T, CC, CI, B, CA, static_cast<long long>(CI) * CA, 64));
  GLF_TRY(make_tmap_bf16(&tmdT, dT, CC, CI, B, CA, static_cast<long long>(CI) * CA, 128));
  GLF_TRY(make_tmap_bf16(&tmS, Sa, CC, CC, B, CA, static_cast<long long>(CA) * CA, 128));
  int dev = 0, num_sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || num_sms <= 0)
    return set_error(GLF_ERR_DEVICE, "gram_wgrad: cannot query the SM count");
  if (num_sms > 160) num_sms = 160;
  // CTAs per product in proportion to its K slabs (theta 4, z 2, g 2, phi 4 per sequence), at least one, at most one
  // per slab
  // (CTA shares 4 : 2 : 2 : 5 — the phi product also forms dt s^T in its epilogue and streams S~ from HBM, measured with
  //  GLF_WGRAD_TRACE: with equal shares per slab its CTAs finished 30 % after the theta / g ones)
  const int w[4] = {4, 2, 2, 4};
  const int share[4] = {4, 2, 2, 5};
  int n[4], used = 0;
  for (int i = 0; i < 4; ++i) {
    long long c = static_cast<long long>(num_sms) * share[i] / 13;
    const long long slabs = static_cast<long long>(w[i]) * B;
    if (c > slabs) c = slabs;
    if (c < 1) c = 1;
    n[i] = static_cast<int>(c);
    used += n[i];
  }
  for (int i = 0; used < num_sms && i < 8; ++i) {   // leftovers to the two large products
    const int k = (i & 1) ? 3 : 0;
    if (n[k] < w[k] * B) { ++n[k]; ++used; }
  }
  WgradParams p;
  p.B = B; p.N = N;
  {
    const char* tr = getenv("GLF_WGRAD_TRACE");
    p.trace = (tr && tr[0] == '1') ? 1 : 0;
  }
  p.cta0[0] = 0;
  for (int i = 0; i < 4; ++i) p.cta0[i + 1] = p.cta0[i] + n[i];
  p.dcv = dcv; p.tv = tv; p.dtv = dtv; p.sfv = sfv;
  p.part = part;
  cudaError_t e = cudaFuncSetAttribute(wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, WG_SMEM);
  if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(wgrad)");
  wgrad_kernel<<<p.cta0[4], WG_THREADS, WG_SMEM, stream>>>(tmWp, tmdQ, tmdWp, tmM, tmdM, tmT, tmdT, tmS, p);
  GLF_TRY(check_cuda(cudaGetLastError(), "wgrad launch"));
  if (p.trace) {
    long long t[4][8];
    cudaStreamSynchronize(stream);
    cudaMemcpyFromSymbol(t, g_wgrad_trace, sizeof(t));
    for (int i = 0; i < 4; ++i)
      fprintf(stderr, "wgrad trace product %d (%d CTAs): mma issued %lld, simt loop done %lld, accumulator ready %lld, partial written %lld cycles after the prologue\n",
              i, n[i], t[i][1] - t[i][0], t[i][2] - t[i][0], t[i][3] - t[i][0], t[i][4] - t[i][0]);
  }
  const int total = 4 * (128 * 256 + 128);
  wgrad_reduce_kernel<<<(total + 255) / 256, 256, 0, stream>>>(part, p.cta0[0], p.cta0[1], p.cta0[2], p.cta0[3],
                                                              p.cta0[4], g->theta_w, g->theta_b, g->wz_w, g->g_w,
                                                              g->g_b, g->phi_w, g->phi_b);
  return check_cuda(cudaGetLastError(), "wgrad_reduce launch");
}

}  // namespace glf
