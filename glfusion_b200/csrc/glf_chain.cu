// glf_chain.cu — the per-sequence [C x C] chain of the Gram form of mode='dot' (R/models/ours.py:866-908 reassociated,
// oracle/tpavi_oracle.py: tpavi_dot_gram_form) as ONE CTA per sequence per direction, C = 256, C' = 128.
//
// Between the token-sized products (S = X^T X, U = X Q^T forward; R = dV^T X, dX = [dV | X][E ; F] backward) every
// sequence owns a chain of [C x C]-sized products.  As separate batched tile GEMMs that chain was 4 launches forward
// and 10 backward per block, each bound by launch + pipeline-fill latency (profiles/r01_v18_launches.csv: 535 us of a
// 1 860 us step).  Here the whole chain of a sequence runs inside one CTA:
//
//   operands      bf16 in shared memory as 64-column SWIZZLE_128B tiles ([rows][64], 128-byte rows) — the layout TMA
//                 writes and tcgen05.mma reads either K-major (K = columns) or MN-major (K = rows), so one copy of a
//                 matrix serves both roles;
//   products      tcgen05.mma, M = 128, fp32 accumulators in TMEM (all 512 columns are used);
//   hand-over     8 drain warps read an accumulator with tcgen05.ld (thread = row), apply the fp32 rank-1 / scale terms
//                 of the homogeneous coordinate, and write bf16 both to global (for the backward / the weight-gradient
//                 products) and straight into the shared-memory tiles of the next product's operand;
//   homogeneous   x~ = [x, 1]: the bias column / row of every augmented matrix is handled in fp32 by the drain threads
//                 (rank-1 updates and matrix-vector products), so the MMAs run on exact C / C' extents.
//
// forward  (chain_fwd_kernel):   T~ = W~phi S~,  M = T~ W~g^T / N,  W' = Wz M^T,  Q~ = W' W~theta
// backward (chain_bwd_kernel):   dQ~ = k2 Q~ S~ + k1 [R | rv] (+ k3 s~^T),  dW' = dQ~ W~theta^T,  dM = dW'^T Wz,
//                                dT~ = dM W~g / N,  F = Wphi^T dT + dT^T Wphi + Q^T k2 Q,  E = k1 Q,  e
// The four weight-gradient sums over the sequences (dW~theta, dWz, dW~g, dW~phi) are NOT formed here: the kernel leaves
// dQ~, dW', dM / N and dT~ in global memory and the caller reduces them with K-concatenated products.
#include <cstdio>
#include <cstdlib>

#include "glf_internal.h"
#include "glf_ptx.cuh"

namespace glf {

namespace {

constexpr int CC = 256;              // channels
constexpr int CI = 128;              // inter channels
constexpr int CA = 264;              // augmented leading dimension (gram_ca(256))
constexpr int CH_DRAIN_WARPS = 8;
constexpr int CH_DRAIN_THREADS = CH_DRAIN_WARPS * 32;
constexpr int CH_THREADS = CH_DRAIN_THREADS + 32;   // + one control warp (TMA producer and MMA issuer)
constexpr uint32_t SLOT = 65536;     // three 64 KB operand slots
constexpr uint32_t Z0 = 0, Z1 = SLOT, Z2 = 2 * SLOT;
constexpr uint32_t VEC_OFF = 3 * SLOT;
constexpr uint32_t VEC_BYTES = 12288;
constexpr uint32_t CH_SMEM = 3 * SLOT + VEC_BYTES + 1024;
constexpr uint32_t BOX_BYTES = 128 * 64 * 2;   // one TMA box: 128 rows x 64 columns

// ---------------------------------------------------------------------------------------------- tile addressing
// matrix held as 64-column tiles of R rows: byte offset of the 16-byte chunk `ch8` (0..7) of `row` inside tile `t`
__device__ __forceinline__ uint32_t tile_chunk(int R, int t, int row, int ch8) {
  return static_cast<uint32_t>(t) * static_cast<uint32_t>(R) * 128u + static_cast<uint32_t>(row) * 128u +
         (static_cast<uint32_t>(ch8 ^ (row & 7)) << 4);
}
// K-major operand descriptor: rows = MN, tiles of 64 K-columns `tile_stride` bytes apart; k16 = K / 16 step
__device__ __forceinline__ uint64_t kdesc(uint32_t base, uint32_t tile_stride, int k16) {
  return make_sdesc(base + static_cast<uint32_t>(k16 >> 2) * tile_stride + static_cast<uint32_t>(k16 & 3) * 32u, 16, 1024);
}
// MN-major operand descriptor: K runs along the rows of the tile (16 rows = 2048 bytes), MN along the columns; the
// next 64-wide MN block is the next tile
__device__ __forceinline__ uint64_t mdesc(uint32_t base, uint32_t tile_stride, int k16) {
  return make_sdesc(base + static_cast<uint32_t>(k16) * 2048u, tile_stride, 1024);
}

// 32 consecutive fp32 values of a row -> bf16 -> shared-memory tile (columns col0 .. col0+31) and global memory
__device__ __forceinline__ void pack32(const float (&f)[32], uint32_t (&pk)[16]) {
#pragma unroll
  for (int j = 0; j < 16; ++j) pk[j] = pack_bf16(f[2 * j], f[2 * j + 1]);
}
__device__ __forceinline__ void st_tile32(uint8_t* mat, int R, int row, int col0, const uint32_t (&pk)[16]) {
  const int t = col0 >> 6, ch0 = (col0 & 63) >> 3;
#pragma unroll
  for (int j = 0; j < 4; ++j)
    *reinterpret_cast<uint4*>(mat + tile_chunk(R, t, row, ch0 + j)) =
        make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
}
__device__ __forceinline__ void st_global32(bf16* dst, const uint32_t (&pk)[16]) {
#pragma unroll
  for (int j = 0; j < 4; ++j)
    *reinterpret_cast<uint4*>(dst + 8 * j) = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
}
__device__ __forceinline__ void ld_acc32(uint32_t taddr, float (&f)[32]) {
  uint32_t v[32];
  tmem_ld_32x32(taddr, v);
  tmem_ld_wait();
#pragma unroll
  for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
}

// dot product of row `row` of a [R x 256] tile matrix with a shared fp32 vector
__device__ __forceinline__ float row_dot256(const uint8_t* mat, int R, int row, const float* vec) {
  float a0 = 0.f, a1 = 0.f;
#pragma unroll 4
  for (int ch = 0; ch < 32; ++ch) {
    const uint4 q = *reinterpret_cast<const uint4*>(mat + tile_chunk(R, ch >> 3, row, ch & 7));
    const uint32_t* q32 = reinterpret_cast<const uint32_t*>(&q);
    const float* v = vec + ch * 8;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const float2 x = unpack_bf16(q32[t]);
      a0 = fmaf(x.x, v[2 * t], a0);
      a1 = fmaf(x.y, v[2 * t + 1], a1);
    }
  }
  return a0 + a1;
}
// acc[0..7] += w * (the 8 bf16 of one 16-byte chunk)
__device__ __forceinline__ void fma_chunk8(const uint8_t* chunk, float w, float (&acc)[8]) {
  const uint4 q = *reinterpret_cast<const uint4*>(chunk);
  const uint32_t* q32 = reinterpret_cast<const uint32_t*>(&q);
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const float2 x = unpack_bf16(q32[t]);
    acc[2 * t] = fmaf(x.x, w, acc[2 * t]);
    acc[2 * t + 1] = fmaf(x.y, w, acc[2 * t + 1]);
  }
}
// element (row, col) of a tile matrix
__device__ __forceinline__ float tile_elem(const uint8_t* mat, int R, int row, int col) {
  return __bfloat162float(
      *reinterpret_cast<const bf16*>(mat + tile_chunk(R, col >> 6, row, (col & 63) >> 3) + (col & 7) * 2));
}

// one 128-row x 64-column box per call; rows row0 .. row0+127 of (batch b) land at dst
__device__ __forceinline__ void load_box(const CUtensorMap* tm, uint32_t bar, uint32_t dst, int col0, int row0, int b) {
  tma_load_4d(tm, bar, dst, col0, row0, b, 0);
}
// [256 x 256] matrix as four [256][64] tiles (32 KB each) at dst
__device__ __forceinline__ void load_256x256(const CUtensorMap* tm, uint32_t bar, uint32_t dst, int b) {
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    load_box(tm, bar, dst + t * 32768u, 64 * t, 0, b);
    load_box(tm, bar, dst + t * 32768u + 16384u, 64 * t, 128, b);
  }
}
// [128 x 256] matrix (rows row0 ..) as four [128][64] tiles (16 KB each) at dst
__device__ __forceinline__ void load_128x256(const CUtensorMap* tm, uint32_t bar, uint32_t dst, int row0, int b) {
#pragma unroll
  for (int t = 0; t < 4; ++t) load_box(tm, bar, dst + t * 16384u, 64 * t, row0, b);
}
// [256 x 128] matrix as two [256][64] tiles at dst; col0 = first column
__device__ __forceinline__ void load_256x128(const CUtensorMap* tm, uint32_t bar, uint32_t dst, int col0, int b) {
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    load_box(tm, bar, dst + t * 32768u, col0 + 64 * t, 0, b);
    load_box(tm, bar, dst + t * 32768u + 16384u, col0 + 64 * t, 128, b);
  }
}

// the mirror image: bulk tensor stores of bf16 tiles that the drain warps left in shared memory
__device__ __forceinline__ void store_256x256(const CUtensorMap* tm, uint32_t src, int row0, int b) {
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    tma_store_4d(tm, src + t * 32768u, 64 * t, row0, b, 0);
    tma_store_4d(tm, src + t * 32768u + 16384u, 64 * t, row0 + 128, b, 0);
  }
}
__device__ __forceinline__ void store_128x256(const CUtensorMap* tm, uint32_t src, int b) {
#pragma unroll
  for (int t = 0; t < 4; ++t) tma_store_4d(tm, src + t * 16384u, 64 * t, 0, b, 0);
}
__device__ __forceinline__ void store_256x128(const CUtensorMap* tm, uint32_t src, int b) {
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    tma_store_4d(tm, src + t * 32768u, 64 * t, 0, b, 0);
    tma_store_4d(tm, src + t * 32768u + 16384u, 64 * t, 128, b, 0);
  }
}
__device__ __forceinline__ void store_128x128(const CUtensorMap* tm, uint32_t src, int b) {
#pragma unroll
  for (int t = 0; t < 2; ++t) tma_store_4d(tm, src + t * 16384u, 64 * t, 0, b, 0);
}

// Debug aid (GLF_CHAIN_TRACE=1): the control thread of CTA 0 records the SM clock each time one of its waits completes;
// the host prints the phase timeline after a stream synchronisation.
__device__ long long g_chain_trace[64];
#define CH_TRACE(i)                                                \
  do {                                                             \
    if (p.trace && blockIdx.x == 0) g_chain_trace[i] = clock64();  \
  } while (0)

constexpr uint32_t IDESC_KK_128 = make_idesc_bf16(128, 128, false, false);
constexpr uint32_t IDESC_KK_256 = make_idesc_bf16(128, 256, false, false);
constexpr uint32_t IDESC_KM_256 = make_idesc_bf16(128, 256, false, true);
constexpr uint32_t IDESC_MM_128 = make_idesc_bf16(128, 128, true, true);
constexpr uint32_t IDESC_MM_256 = make_idesc_bf16(128, 256, true, true);

struct ChainFwdParams {
  int N;
  const float *sfv, *bphi, *bg, *bth;   // s [B][C]; biases [C'] fp32
  bf16 *T, *Mb, *Wp, *Qb;               // T~ [B][C'][Ca], M [B][C'][C'], W' [B][C][C'], Q~ [B][C][Ca]
  float* cvec;                          // c = W' b_theta  [B][C]
  float* tv;                            // t = T~[:, C]    [B][C'] (fp32 copy for the weight-gradient kernel)
};

// ---------------------------------------------------------------------------------------------- forward chain
//   F1  T  = Wphi S   (+ bphi s^T)          [128 x 256]   A = Wphi (K-major), B = S (symmetric: K-major)
//       t  = Wphi s + N bphi                               (fp32, drain threads)
//   F2  M  = (T Wg^T + t bg^T) / N          [128 x 128]   A = T, B = Wg (K-major)
//   F3  W' = Wz M^T                         [256 x 128]   A = Wz, B = M (K-major)
//   F4  Q  = W' Wtheta ,  c = W' btheta     [256 x 256]   A = W' (K-major), B = Wtheta (MN-major)
__global__ void __launch_bounds__(CH_THREADS, 1)
    chain_fwd_kernel(const __grid_constant__ CUtensorMap tmS, const __grid_constant__ CUtensorMap tmW,
                     const __grid_constant__ CUtensorMap tmWz, const __grid_constant__ CUtensorMap tmT,
                     const __grid_constant__ CUtensorMap tmM, const __grid_constant__ CUtensorMap tmWp,
                     const __grid_constant__ CUtensorMap tmQ, const ChainFwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sgen = smem_raw + (sbase - smem_u32(smem_raw));
  float* v_s = reinterpret_cast<float*>(sgen + VEC_OFF);   // [256]
  float* v_bphi = v_s + 256;                               // [128]
  float* v_bg = v_bphi + 128;
  float* v_bth = v_bg + 128;
  float* v_t = v_bth + 128;                                // [128]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sgen + VEC_OFF + 8192);
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(sgen + VEC_OFF + 8192 + 256);
  enum { LD0 = 0, LD1, LD2, LD3, MMA0, MMA1, MMA2, MMA3, DR0, DR1, DR2, DR3, NBAR };
  auto bar = [&](int i) { return smem_u32(&bars[i]); };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x;
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmS);
    tma_prefetch_desc(&tmW);
    tma_prefetch_desc(&tmWz);
    for (int i = 0; i < NBAR; ++i) mbar_init(bar(i), (i >= DR0) ? CH_DRAIN_WARPS : 1);
    fence_mbar_init();
  }
  if (warp == CH_DRAIN_WARPS) tmem_alloc(smem_u32(tmem_holder), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_holder;

  if (warp == CH_DRAIN_WARPS) {
    // ------------------------------------------------------------------------------------------ control warp
    if (elect_one()) {
      mbar_expect_tx(bar(LD0), 12 * BOX_BYTES);
      load_256x256(&tmS, bar(LD0), sbase + Z0, b);             // S -> Z0, Z1
      load_128x256(&tmW, bar(LD0), sbase + Z2, CI, 0);         // Wphi -> Z2
      mbar_wait(bar(LD0), 0);
      tc_fence_after();
      for (int k = 0; k < 16; ++k)
        umma_f16(tmem, kdesc(sbase + Z2, 16384, k), kdesc(sbase + Z0, 32768, k), IDESC_KK_256, k > 0);
      umma_commit(bar(MMA0));
      mbar_wait(bar(MMA0), 0);                                  // S and Wphi are dead
      mbar_expect_tx(bar(LD1), 4 * BOX_BYTES);
      load_128x256(&tmW, bar(LD1), sbase + Z0, 2 * CI, 0);     // Wg -> Z0
      mbar_expect_tx(bar(LD2), 4 * BOX_BYTES);
      load_256x128(&tmWz, bar(LD2), sbase + Z1, 0, 0);         // Wz -> Z1
      mbar_wait(bar(DR0), 0);                                   // T (bf16) in Z2
      store_128x256(&tmT, sbase + Z2, b);
      tma_store_commit();
      mbar_wait(bar(LD1), 0);
      tc_fence_after();
      for (int k = 0; k < 16; ++k)
        umma_f16(tmem + 256, kdesc(sbase + Z2, 16384, k), kdesc(sbase + Z0, 16384, k), IDESC_KK_128, k > 0);
      umma_commit(bar(MMA1));
      mbar_wait(bar(MMA1), 0);                                  // T and Wg are dead
      tma_store_wait_read<0>();                                 // ... and the store of T has read Z2
      mbar_expect_tx(bar(LD3), 4 * BOX_BYTES);
      load_128x256(&tmW, bar(LD3), sbase + Z2, 0, 0);          // Wtheta -> Z2
      mbar_wait(bar(DR1), 0);                                   // M (bf16) in Z0
      store_128x128(&tmM, sbase + Z0, b);
      tma_store_commit();
      mbar_wait(bar(LD2), 0);
      tc_fence_after();
      for (int h = 0; h < 2; ++h)
        for (int k = 0; k < 8; ++k)
          umma_f16(tmem + h * 128, kdesc(sbase + Z1 + h * 16384, 32768, k), kdesc(sbase + Z0, 16384, k), IDESC_KK_128,
                   k > 0);
      tma_store_wait_read<0>();      // before the accumulator is published: the drain of W' overwrites M in Z0
      umma_commit(bar(MMA2));
      mbar_wait(bar(DR2), 0);                                   // W' (bf16) in Z0
      store_256x128(&tmWp, sbase + Z0, b);
      tma_store_commit();
      mbar_wait(bar(LD3), 0);
      tc_fence_after();
      for (int h = 0; h < 2; ++h)
        for (int k = 0; k < 8; ++k)
          umma_f16(tmem + h * 256, kdesc(sbase + Z0 + h * 16384, 32768, k), mdesc(sbase + Z2, 16384, k), IDESC_KM_256,
                   k > 0);
      umma_commit(bar(MMA3));
      mbar_wait(bar(DR3), 0);                                   // Q (bf16) in Z1, Z2
      store_256x256(&tmQ, sbase + Z1, 0, b);
      tma_store_commit();
      tma_store_wait_all<0>();
    }
  } else {
    // ------------------------------------------------------------------------------------------ drain warps
    const int tid = threadIdx.x;            // 0..255
    const int q = warp & 3, hf = warp >> 2;
    const uint32_t tlane = tmem + (static_cast<uint32_t>(q * 32) << 16);
    const float fN = static_cast<float>(p.N), invN = 1.f / fN;
    v_s[tid] = p.sfv[static_cast<long long>(b) * CC + tid];
    if (tid < CI) {
      v_bphi[tid] = p.bphi[tid];
      v_bg[tid] = p.bg[tid];
      v_bth[tid] = p.bth[tid];
    }
    named_bar_sync(1, CH_DRAIN_THREADS);
    mbar_wait(bar(LD0), 0);
    if (tid < CI) {
      v_t[tid] = fmaf(fN, v_bphi[tid], row_dot256(sgen + Z2, 128, tid, v_s));
      p.tv[static_cast<long long>(b) * CI + tid] = v_t[tid];
    }
    named_bar_sync(1, CH_DRAIN_THREADS);
    // ---- T = acc + bphi s^T  -> Z2 ([128][64] x 4) and global
    mbar_wait(bar(MMA0), 0);
    tc_fence_after();
    {
      const int i = q * 32 + lane;
      const float bp = v_bphi[i];
      bf16* Trow = p.T + (static_cast<long long>(b) * CI + i) * CA;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        const int col0 = hf * 128 + c * 32;
        float f[32];
        ld_acc32(tlane + col0, f);
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = fmaf(bp, v_s[col0 + j], f[j]);
        uint32_t pk[16];
        pack32(f, pk);
        st_tile32(sgen + Z2, 128, i, col0, pk);
      }
      if (hf == 1) *reinterpret_cast<uint4*>(Trow + CC) = make_uint4(pack_bf16(v_t[i], 0.f), 0u, 0u, 0u);
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar(DR0));
    // ---- M = (acc + t bg^T) / N  -> Z0 ([128][64] x 2) and global
    mbar_wait(bar(MMA1), 0);
    tc_fence_after();
    {
      const int i = q * 32 + lane;
      const float ti = v_t[i];
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        const int col0 = hf * 64 + c * 32;
        float f[32];
        ld_acc32(tlane + 256 + col0, f);
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = fmaf(ti, v_bg[col0 + j], f[j]) * invN;
        uint32_t pk[16];
        pack32(f, pk);
        st_tile32(sgen + Z0, 128, i, col0, pk);
      }
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar(DR1));
    // ---- W' -> Z0 ([256][64] x 2) and global; c = W' btheta
    const int r = hf * 128 + q * 32 + lane;     // row of W' / Q owned by this thread
    float cv = 0.f;
    mbar_wait(bar(MMA2), 0);
    tc_fence_after();
    {
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        const int col0 = c * 32;
        float f[32];
        ld_acc32(tlane + hf * 128 + col0, f);
        uint32_t pk[16];
        pack32(f, pk);
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float2 x = unpack_bf16(pk[j]);
          cv = fmaf(x.x, v_bth[col0 + 2 * j], cv);
          cv = fmaf(x.y, v_bth[col0 + 2 * j + 1], cv);
        }
        st_tile32(sgen + Z0, 256, r, col0, pk);
      }
      p.cvec[static_cast<long long>(b) * CC + r] = cv;
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar(DR2));
    // ---- Q~ -> global
    mbar_wait(bar(MMA3), 0);
    tc_fence_after();
    {
      bf16* Qrow = p.Qb + (static_cast<long long>(b) * CC + r) * CA;
#pragma unroll 1
      for (int c = 0; c < 8; ++c) {
        const int col0 = c * 32;
        float f[32];
        ld_acc32(tlane + hf * 256 + col0, f);
        uint32_t pk[16];
        pack32(f, pk);
        st_tile32(sgen + Z1, 256, r, col0, pk);
      }
      *reinterpret_cast<uint4*>(Qrow + CC) = make_uint4(pack_bf16(cv, 0.f), 0u, 0u, 0u);
    }
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar(DR3));
  }
  tc_fence_before();
  __syncthreads();
  if (warp == CH_DRAIN_WARPS) tmem_dealloc(tmem, 512);
}

struct ChainBwdParams {
  int N, has_k2, trace;
  const float *sfv, *cvec, *rv, *k1, *k2, *k3;   // s, c, rv [B][C]; BatchNorm-backward coefficients [C]
  const float *bth, *bphi, *bg;                  // biases [C'] fp32
  const bf16* Rb;                                // [B][Ca][Ca]: rows < C hold k1 [R | rv]
  bf16 *dQa, *dWp, *dMn, *dT, *EF;               // dQ~ [B][C][Ca], dW' [B][C][C'], dM/N [B][C'][C'], dT~ [B][C'][Ca], [E;F] [B][2C][C]
  float* evec;                                   // e [B][C]
  float *dcv, *dtv;                              // fp32 copies of dQ~[:, C] [B][C] and dT~[:, C] [B][C'] (weight gradients)
};

// ---------------------------------------------------------------------------------------------- backward chain
//   B1  QS = Q S                            [256 x 256]   A = Q (K-major), B = S in two 128-row halves
//       dQ = k1 R + k2 QS + (k2 c + k3) s^T ;  dc = k1 rv + k2 (Q s + N c) + N k3 ;  E = k1 Q
//   B2  dW' = dQ Wtheta^T + dc btheta^T     [256 x 128]   A = dQ, B = Wtheta (K-major)
//   B5  dM = dW'^T Wz                       [128 x 128]   A = dW' (MN-major), B = Wz (MN-major)
//   B6  dT = (dM / N) Wg ,  dt = (dM / N) bg   [128 x 256]   A = dM / N (K-major), B = Wg (MN-major)
//   B9  F = Wphi^T dT + dT^T Wphi + Q^T (k2 Q)   [256 x 256]   all operands MN-major, one accumulator
//       e = Wphi^T dt + dT^T bphi + Q^T (k2 c + k3)
__global__ void __launch_bounds__(CH_THREADS, 1)
    chain_bwd_kernel(const __grid_constant__ CUtensorMap tmS, const __grid_constant__ CUtensorMap tmQ,
                     const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmWz,
                     const __grid_constant__ CUtensorMap tmdQ, const __grid_constant__ CUtensorMap tmdWp,
                     const __grid_constant__ CUtensorMap tmdM, const __grid_constant__ CUtensorMap tmdT,
                     const __grid_constant__ CUtensorMap tmEF, const __grid_constant__ CUtensorMap tmR,
                     const ChainBwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sgen = smem_raw + (sbase - smem_u32(smem_raw));
  float* v_s = reinterpret_cast<float*>(sgen + VEC_OFF);   // [256]
  float* v_k1 = v_s + 256;
  float* v_k2 = v_k1 + 256;
  float* v_v = v_k2 + 256;        // k2 c + k3
  float* v_dc = v_v + 256;
  float* v_e = v_dc + 256;        // e accumulates here
  float* v_bth = v_e + 256;       // [128]
  float* v_bphi = v_bth + 128;
  float* v_bg = v_bphi + 128;
  float* v_dt = v_bg + 128;       // [2][128] partial, then [128]   (the vectors end at byte 8704)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sgen + VEC_OFF + 10240);
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(sgen + VEC_OFF + 10240 + 256);
  static_assert(10240 + 256 + 16 <= VEC_BYTES, "vector area");
  enum { LDA = 0, LDB, LDC, LDD, LDE, LDF, LDG, LDH, MMAA, MMAB, MMAC, MMAD, MMAE, MMAF, MMAG0, MMAG1,
         LDR, DRA, DRB, DRC, DRD, DRE, DRK0, DRK1, DRF, DRQ, NBAR };
  auto bar = [&](int i) { return smem_u32(&bars[i]); };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x;
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmS);
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmW);
    tma_prefetch_desc(&tmWz);
    for (int i = 0; i < NBAR; ++i) mbar_init(bar(i), (i >= DRA) ? CH_DRAIN_WARPS : 1);
    fence_mbar_init();
    tma_prefetch_desc(&tmR);
  }
  if (warp == CH_DRAIN_WARPS) tmem_alloc(smem_u32(tmem_holder), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_holder;

  if (warp == CH_DRAIN_WARPS) {
    // ------------------------------------------------------------------------------------------ control warp
    if (elect_one()) {
      CH_TRACE(0);
      mbar_expect_tx(bar(LDA), 12 * BOX_BYTES);
      load_256x256(&tmQ, bar(LDA), sbase + Z0, b);             // Q -> Z0, Z1
      load_128x256(&tmS, bar(LDA), sbase + Z2, 0, b);          // S rows 0..127 -> Z2
      mbar_wait(bar(LDA), 0); CH_TRACE(1);
      tc_fence_after();
      for (int h = 0; h < 2; ++h)
        for (int k = 0; k < 16; ++k)
          umma_f16(tmem + h * 256, kdesc(sbase + Z0 + h * 16384, 32768, k), kdesc(sbase + Z2, 16384, k), IDESC_KK_128,
                   k > 0);
      umma_commit(bar(MMAA));
      mbar_wait(bar(MMAA), 0); CH_TRACE(2);
      mbar_expect_tx(bar(LDB), 4 * BOX_BYTES);
      load_128x256(&tmS, bar(LDB), sbase + Z2, 128, b);        // S rows 128..255 -> Z2
      mbar_wait(bar(LDB), 0); CH_TRACE(3);
      tc_fence_after();
      for (int h = 0; h < 2; ++h)
        for (int k = 0; k < 16; ++k)
          umma_f16(tmem + h * 256 + 128, kdesc(sbase + Z0 + h * 16384, 32768, k), kdesc(sbase + Z2, 16384, k),
                   IDESC_KK_128, k > 0);
      umma_commit(bar(MMAB));
      mbar_wait(bar(MMAB), 0); CH_TRACE(4);
      mbar_wait(bar(DRQ), 0);                                   // the drain warps have finished reading Q (Q s, E)
      mbar_expect_tx(bar(LDR), 8 * BOX_BYTES);
      load_256x256(&tmR, bar(LDR), sbase + Z0, b);             // k1 R -> Z0, Z1: dQ is formed in place on top of it
      mbar_expect_tx(bar(LDC), 4 * BOX_BYTES);
      load_128x256(&tmW, bar(LDC), sbase + Z2, 0, 0);          // Wtheta -> Z2
      mbar_wait(bar(DRA), 0); CH_TRACE(5);                                   // dQ (bf16) in Z0, Z1
      store_256x256(&tmdQ, sbase + Z0, 0, b);
      tma_store_commit();
      mbar_wait(bar(LDC), 0); CH_TRACE(6);
      tc_fence_after();
      for (int h = 0; h < 2; ++h)
        for (int k = 0; k < 16; ++k)
          umma_f16(tmem + h * 128, kdesc(sbase + Z0 + h * 16384, 32768, k), kdesc(sbase + Z2, 16384, k), IDESC_KK_128,
                   k > 0);
      tma_store_wait_read<0>();      // before the accumulator is published: the drain of dW' overwrites dQ in Z0
      umma_commit(bar(MMAC));
      mbar_wait(bar(MMAC), 0); CH_TRACE(7);
      mbar_expect_tx(bar(LDD), 4 * BOX_BYTES);
      load_256x128(&tmWz, bar(LDD), sbase + Z2, 0, 0);         // Wz -> Z2
      mbar_wait(bar(DRB), 0); CH_TRACE(8);                                   // dW' (bf16) in Z0
      store_256x128(&tmdWp, sbase + Z0, b);
      tma_store_commit();
      mbar_wait(bar(LDD), 0); CH_TRACE(9);
      tc_fence_after();
      for (int k = 0; k < 16; ++k)
        umma_f16(tmem + 256, mdesc(sbase + Z0, 32768, k), mdesc(sbase + Z2, 32768, k), IDESC_MM_128, k > 0);
      tma_store_wait_read<0>();
      umma_commit(bar(MMAD));
      mbar_wait(bar(MMAD), 0); CH_TRACE(10);
      mbar_expect_tx(bar(LDE), 4 * BOX_BYTES);
      load_128x256(&tmW, bar(LDE), sbase + Z1, 2 * CI, 0);     // Wg -> Z1
      mbar_expect_tx(bar(LDF), 4 * BOX_BYTES);
      load_128x256(&tmW, bar(LDF), sbase + Z2, CI, 0);         // Wphi -> Z2
      mbar_wait(bar(DRC), 0); CH_TRACE(11);                                   // dM / N (bf16) in Z0
      store_128x128(&tmdM, sbase + Z0, b);
      tma_store_commit();
      mbar_wait(bar(LDE), 0); CH_TRACE(12);
      tc_fence_after();
      for (int k = 0; k < 8; ++k)
        umma_f16(tmem, kdesc(sbase + Z0, 16384, k), mdesc(sbase + Z1, 16384, k), IDESC_KM_256, k > 0);
      tma_store_wait_read<0>();
      umma_commit(bar(MMAE));
      mbar_wait(bar(MMAE), 0); CH_TRACE(13);
      if (p.has_k2) {
        mbar_expect_tx(bar(LDG), 4 * BOX_BYTES);
        load_256x128(&tmQ, bar(LDG), sbase + Z1, 0, b);        // Q columns 0..127 -> Z1
      }
      mbar_wait(bar(DRD), 0); CH_TRACE(14);                                   // dT (bf16) in Z0
      store_128x256(&tmdT, sbase + Z0, b);
      tma_store_commit();
      mbar_wait(bar(LDF), 0); CH_TRACE(15);
      tc_fence_after();
      for (int h = 0; h < 2; ++h) {
        for (int k = 0; k < 8; ++k)
          umma_f16(tmem + h * 256, mdesc(sbase + Z2 + h * 32768, 16384, k), mdesc(sbase + Z0, 16384, k), IDESC_MM_256,
                   k > 0);
        for (int k = 0; k < 8; ++k)
          umma_f16(tmem + h * 256, mdesc(sbase + Z0 + h * 32768, 16384, k), mdesc(sbase + Z2, 16384, k), IDESC_MM_256, 1);
      }
      tma_store_wait_read<0>();      // dT has been stored before anything (drain of F, next Q half) overwrites Z0
      umma_commit(bar(MMAF));
      if (p.has_k2) {
        mbar_wait(bar(MMAF), 0); CH_TRACE(16);
        mbar_wait(bar(DRE), 0); CH_TRACE(17);                                 // the e terms that read dT / Wphi are done
        mbar_expect_tx(bar(LDH), 4 * BOX_BYTES);
        load_256x128(&tmQ, bar(LDH), sbase + Z0, 128, b);      // Q columns 128..255 -> Z0
        mbar_wait(bar(LDH), 0); CH_TRACE(18);
        for (int g = 0; g < 2; ++g) {
          mbar_wait(bar(DRK0 + g), 0); CH_TRACE(19 + g);                          // k2 Q[:, 128 g ..] in Z2
          tc_fence_after();
          for (int h = 0; h < 2; ++h)
            for (int k = 0; k < 16; ++k)
              umma_f16(tmem + h * 256 + g * 128, mdesc(sbase + (h == 0 ? Z1 : Z0), 32768, k),
                       mdesc(sbase + Z2, 32768, k), IDESC_MM_128, 1);
          umma_commit(bar(MMAG0 + g));
        }
      }
      mbar_wait(bar(DRF), 0); CH_TRACE(21);                                   // F (bf16) in Z0, Z1
      store_256x256(&tmEF, sbase + Z0, CC, b);
      tma_store_commit();
      tma_store_wait_all<0>();
    }
  } else {
    // ------------------------------------------------------------------------------------------ drain warps
    const int tid = threadIdx.x;            // 0..255
    const int q = warp & 3, hf = warp >> 2;
    const uint32_t tlane = tmem + (static_cast<uint32_t>(q * 32) << 16);
    const float fN = static_cast<float>(p.N), invN = 1.f / fN;
    const long long bC = static_cast<long long>(b) * CC;
    const float my_c = p.cvec[bC + tid];
    {
      const float a1 = p.k1[tid], a2 = p.k2[tid], a3 = p.k3[tid];
      v_s[tid] = p.sfv[bC + tid];
      v_k1[tid] = a1;
      v_k2[tid] = a2;
      v_v[tid] = fmaf(a2, my_c, a3);
      v_e[tid] = 0.f;
      if (tid < CI) {
        v_bth[tid] = p.bth[tid];
        v_bphi[tid] = p.bphi[tid];
        v_bg[tid] = p.bg[tid];
      }
    }
    named_bar_sync(1, CH_DRAIN_THREADS);
    mbar_wait(bar(LDA), 0);
    {
      // dc = k1 rv + k2 (Q s + N c) + N k3       (thread = row of Q)
      const float qs = row_dot256(sgen + Z0, 256, tid, v_s);
      v_dc[tid] = fmaf(v_k1[tid], p.rv[bC + tid], fmaf(v_k2[tid], fmaf(fN, my_c, qs), fN * p.k3[tid]));
      p.dcv[bC + tid] = v_dc[tid];
      // E' = k1 Q + I -> EF[b][0]   (a warp moves one 512-byte row per iteration).  The residual dV of
      // dX = dV E + X F + 1 e^T + dV is folded into the first operand (one more bf16 rounding of the 256 diagonal entries:
      // <= 2^-9 |dV_j| on dX_j, an order below the bf16 rounding of dX itself), so the dX GEMM needs no addend pass over
      // dV in its epilogue and its tiles leave through bulk tensor stores.
      bf16* E = p.EF + static_cast<long long>(b) * 2 * CC * CC;
#pragma unroll 2
      for (int it = 0; it < 32; ++it) {
        const int row = it * 8 + warp;
        const float a1 = v_k1[row];
        const uint4 qv = *reinterpret_cast<const uint4*>(sgen + Z0 + tile_chunk(256, lane >> 3, row, lane & 7));
        const uint32_t* q32 = reinterpret_cast<const uint32_t*>(&qv);
        uint32_t o[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const float2 x = unpack_bf16(q32[t]);
          const int col = lane * 8 + 2 * t;
          o[t] = pack_bf16(a1 * x.x + (col == row ? 1.f : 0.f), a1 * x.y + (col + 1 == row ? 1.f : 0.f));
        }
        *reinterpret_cast<uint4*>(E + static_cast<long long>(row) * CC + lane * 8) = make_uint4(o[0], o[1], o[2], o[3]);
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(bar(DRQ));     // every reader of Q (Z0, Z1) is done before k1 R is loaded on top of it
    named_bar_sync(1, CH_DRAIN_THREADS);      // v_dc is read by other threads below
    const int r = hf * 128 + q * 32 + lane;   // row of the 256-row matrices owned by this thread
    // ---- dQ = k1 R + k2 QS + v s^T  -> Z0, Z1 ([256][64] x 4), stored by the control thread
    {
      // k1 R was brought into Z0 / Z1 by TMA in the layout dQ takes: every thread reads its own 64 bytes of a chunk
      // and writes the result back to the same place
      mbar_wait(bar(MMAB), 0);
      mbar_wait(bar(LDR), 0);
      tc_fence_after();
      const float a2 = v_k2[r], vr = v_v[r];
      bf16* Drow = p.dQa + (bC + r) * CA;
#pragma unroll 1
      for (int c = 0; c < 8; ++c) {
        const int col0 = c * 32;
        float f[32];
        ld_acc32(tlane + hf * 256 + col0, f);
        uint8_t* tile = sgen + Z0;
        const int t = col0 >> 6, ch0 = (col0 & 63) >> 3;
        uint4 rk[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) rk[j] = *reinterpret_cast<const uint4*>(tile + tile_chunk(256, t, r, ch0 + j));
        const uint32_t* r32 = reinterpret_cast<const uint32_t*>(rk);
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float2 x = unpack_bf16(r32[j]);
          f[2 * j] = fmaf(a2, f[2 * j], fmaf(vr, v_s[col0 + 2 * j], x.x));
          f[2 * j + 1] = fmaf(a2, f[2 * j + 1], fmaf(vr, v_s[col0 + 2 * j + 1], x.y));
        }
        uint32_t pk[16];
        pack32(f, pk);
        st_tile32(sgen + Z0, 256, r, col0, pk);
      }
      *reinterpret_cast<uint4*>(Drow + CC) = make_uint4(pack_bf16(v_dc[r], 0.f), 0u, 0u, 0u);
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar(DRA));
    // ---- dW' = acc + dc btheta^T  -> Z0 ([256][64] x 2) and global
    mbar_wait(bar(MMAC), 0);
    tc_fence_after();
    {
      const float dcr = v_dc[r];
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        const int col0 = c * 32;
        float f[32];
        ld_acc32(tlane + hf * 128 + col0, f);
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = fmaf(dcr, v_bth[col0 + j], f[j]);
        uint32_t pk[16];
        pack32(f, pk);
        st_tile32(sgen + Z0, 256, r, col0, pk);
      }
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar(DRB));
    // ---- dM / N  -> Z0 ([128][64] x 2) and global;  dt = (dM / N) bg
    mbar_wait(bar(MMAD), 0);
    tc_fence_after();
    {
      const int i = q * 32 + lane;
      float dtp = 0.f;
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        const int col0 = hf * 64 + c * 32;
        float f[32];
        ld_acc32(tlane + 256 + col0, f);
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] *= invN;
        uint32_t pk[16];
        pack32(f, pk);
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float2 x = unpack_bf16(pk[j]);
          dtp = fmaf(x.x, v_bg[col0 + 2 * j], dtp);
          dtp = fmaf(x.y, v_bg[col0 + 2 * j + 1], dtp);
        }
        st_tile32(sgen + Z0, 128, i, col0, pk);
      }
      v_dt[hf * 128 + i] = dtp;
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar(DRC));
    named_bar_sync(1, CH_DRAIN_THREADS);
    float my_dt = 0.f;
    if (tid < CI) my_dt = v_dt[tid] + v_dt[128 + tid];
    named_bar_sync(1, CH_DRAIN_THREADS);
    if (tid < CI) {
      v_dt[tid] = my_dt;
      p.dtv[static_cast<long long>(b) * CI + tid] = my_dt;
    }
    named_bar_sync(1, CH_DRAIN_THREADS);
    // ---- dT -> Z0 ([128][64] x 4) and global (column C = dt)
    mbar_wait(bar(MMAE), 0);
    tc_fence_after();
    {
      const int i = q * 32 + lane;
      bf16* Trow = p.dT + (static_cast<long long>(b) * CI + i) * CA;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        const int col0 = hf * 128 + c * 32;
        float f[32];
        ld_acc32(tlane + col0, f);
        uint32_t pk[16];
        pack32(f, pk);
        st_tile32(sgen + Z0, 128, i, col0, pk);
      }
      if (hf == 1) *reinterpret_cast<uint4*>(Trow + CC) = make_uint4(pack_bf16(v_dt[i], 0.f), 0u, 0u, 0u);
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar(DRD));
    named_bar_sync(1, CH_DRAIN_THREADS);      // dT complete in Z0 for the column reads below
    // ---- e  = Wphi^T dt + dT^T bphi     (thread = column m; Wphi in Z2, dT in Z0, both [128][64] x 4)
    mbar_wait(bar(LDF), 0);
    {
      // a warp owns four 8-column chunks; lane = (chunk sub = lane / 8, row residue rl = lane % 8): 16 rows x 8 columns
      // of both matrices per lane, then a shuffle reduction over the eight row residues
      const int cc = warp * 4 + (lane >> 3), rl = lane & 7;
      float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
      for (int i = rl; i < CI; i += 8) {
        const uint32_t off = tile_chunk(128, cc >> 3, i, cc & 7);
        fma_chunk8(sgen + Z2 + off, v_dt[i], acc);
        fma_chunk8(sgen + Z0 + off, v_bphi[i], acc);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 1);
        acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 2);
        acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 4);
      }
      if (rl == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) v_e[cc * 8 + j] = acc[j];
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(bar(DRE));
    named_bar_sync(1, CH_DRAIN_THREADS);      // v_e is complete before its owners change below
    if (p.has_k2) {
      // ---- k2 Q[:, 128 g .. 128 g + 127] -> Z2 ([256][64] x 2);  e += Q^T (k2 c + k3)
      mbar_wait(bar(MMAF), 0);                // Wphi (Z2) has been consumed
      for (int g = 0; g < 2; ++g) {
        mbar_wait(bar(g == 0 ? LDG : LDH), 0);
        if (g == 1) mbar_wait(bar(MMAG0), 0); // the previous half of k2 Q has been consumed
        const uint8_t* src = sgen + (g == 0 ? Z1 : Z0);
        // (small unroll factors throughout: every phase of this kernel runs once, so its code is fetched cold and a
        // long unrolled body costs more in instruction-cache misses than it saves in issue slots)
#pragma unroll 2
        for (int it = 0; it < 16; ++it) {
          const int idx = it * CH_DRAIN_THREADS + tid;      // 2 tiles x 256 rows x 8 chunks
          const int row = (idx >> 3) & 255;
          const uint32_t off = static_cast<uint32_t>(idx) * 16u;   // same swizzled position in source and destination
          const float a2 = v_k2[row];
          const uint4 qv = *reinterpret_cast<const uint4*>(src + off);
          const uint32_t* q32 = reinterpret_cast<const uint32_t*>(&qv);
          uint32_t o[4];
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const float2 x = unpack_bf16(q32[t]);
            o[t] = pack_bf16(a2 * x.x, a2 * x.y);
          }
          *reinterpret_cast<uint4*>(sgen + Z2 + off) = make_uint4(o[0], o[1], o[2], o[3]);
        }
        {
          // a warp owns two 8-column chunks of this half of Q; lane = (chunk sub = lane / 16, row residue rl = lane % 16)
          const int cc = warp * 2 + (lane >> 4), rl = lane & 15;
          float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
          for (int i = rl; i < CC; i += 16) fma_chunk8(src + tile_chunk(256, cc >> 3, i, cc & 7), v_v[i], acc);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 1);
            acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 2);
            acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 4);
            acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 8);
          }
          if (rl == 0) {
#pragma unroll
            for (int j = 0; j < 8; ++j) v_e[g * 128 + cc * 8 + j] += acc[j];
          }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(DRK0 + g));
      }
    }
    // ---- F -> EF[b][1]
    mbar_wait(bar(p.has_k2 ? MMAG1 : MMAF), 0);
    tc_fence_after();
    {
#pragma unroll 1
      for (int c = 0; c < 8; ++c) {
        const int col0 = c * 32;
        float f[32];
        ld_acc32(tlane + hf * 256 + col0, f);
        uint32_t pk[16];
        pack32(f, pk);
        st_tile32(sgen + Z0, 256, r, col0, pk);
      }
    }
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar(DRF));
    named_bar_sync(1, CH_DRAIN_THREADS);
    p.evec[bC + tid] = v_e[tid];
  }
  tc_fence_before();
  __syncthreads();
  if (warp == CH_DRAIN_WARPS) tmem_dealloc(tmem, 512);
}

}  // namespace

bool gram_chain_supported(int C, int Ci) {
  if (const char* e = getenv("GLF_GRAM_CHAIN")) {   // tuning aid: GLF_GRAM_CHAIN=0 keeps the batched tile GEMMs
    if (e[0] == '0') return false;
  }
  return C == CC && Ci == CI;
}

int gram_chain_fwd(const bf16* Sa, const float* sfv, const bf16* waug, const bf16* wz, const float* bphi,
                   const float* bg, const float* bth, bf16* T, bf16* Mb, bf16* Wp, bf16* Qb, float* cvec, float* tv, int B,
                   int N, cudaStream_t stream) {
  CUtensorMap tmS, tmW, tmWz, tmT, tmM, tmWp, tmQ;
  GLF_TRY(make_tmap_bf16(&tmS, Sa, CC, CC, B, CA, static_cast<long long>(CA) * CA, 128));
  GLF_TRY(make_tmap_bf16(&tmW, waug, CC, 3 * CI, 1, CA, 0, 128));
  GLF_TRY(make_tmap_bf16(&tmWz, wz, CI, CC, 1, CI, 0, 128));
  GLF_TRY(make_tmap_bf16(&tmT, T, CC, CI, B, CA, static_cast<long long>(CI) * CA, 128));
  GLF_TRY(make_tmap_bf16(&tmM, Mb, CI, CI, B, CI, static_cast<long long>(CI) * CI, 128));
  GLF_TRY(make_tmap_bf16(&tmWp, Wp, CI, CC, B, CI, static_cast<long long>(CC) * CI, 128));
  GLF_TRY(make_tmap_bf16(&tmQ, Qb, CC, CC, B, CA, static_cast<long long>(CC) * CA, 128));
  ChainFwdParams p;
  p.N = N;
  p.sfv = sfv; p.bphi = bphi; p.bg = bg; p.bth = bth;
  p.T = T; p.Mb = Mb; p.Wp = Wp; p.Qb = Qb; p.cvec = cvec; p.tv = tv;
  cudaError_t e = cudaFuncSetAttribute(chain_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CH_SMEM);
  if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(chain_fwd)");
  chain_fwd_kernel<<<B, CH_THREADS, CH_SMEM, stream>>>(tmS, tmW, tmWz, tmT, tmM, tmWp, tmQ, p);
  return check_cuda(cudaGetLastError(), "chain_fwd launch");
}

int gram_chain_bwd(const bf16* Sa, const bf16* Qb, const bf16* waug, const bf16* wz, const bf16* Rb, const float* sfv,
                   const float* cvec, const float* rv, const float* k1, const float* k2, const float* k3,
                   const float* bth, const float* bphi, const float* bg, int has_k2, bf16* dQa, bf16* dWp, bf16* dMn,
                   bf16* dT, bf16* EF, float* evec, float* dcv, float* dtv, int B, int N, cudaStream_t stream) {
  CUtensorMap tmS, tmQ, tmW, tmWz;
  GLF_TRY(make_tmap_bf16(&tmS, Sa, CC, CC, B, CA, static_cast<long long>(CA) * CA, 128));
  GLF_TRY(make_tmap_bf16(&tmQ, Qb, CC, CC, B, CA, static_cast<long long>(CC) * CA, 128));
  GLF_TRY(make_tmap_bf16(&tmW, waug, CC, 3 * CI, 1, CA, 0, 128));
  GLF_TRY(make_tmap_bf16(&tmWz, wz, CI, CC, 1, CI, 0, 128));
  CUtensorMap tmdQ, tmdWp, tmdM, tmdT, tmEF, tmR;
  GLF_TRY(make_tmap_bf16(&tmR, Rb, CC, CC, B, CA, static_cast<long long>(CA) * CA, 128));
  GLF_TRY(make_tmap_bf16(&tmdQ, dQa, CC, CC, B, CA, static_cast<long long>(CC) * CA, 128));
  GLF_TRY(make_tmap_bf16(&tmdWp, dWp, CI, CC, B, CI, static_cast<long long>(CC) * CI, 128));
  GLF_TRY(make_tmap_bf16(&tmdM, dMn, CI, CI, B, CI, static_cast<long long>(CI) * CI, 128));
  GLF_TRY(make_tmap_bf16(&tmdT, dT, CC, CI, B, CA, static_cast<long long>(CI) * CA, 128));
  GLF_TRY(make_tmap_bf16(&tmEF, EF, CC, 2 * CC, B, CC, 2LL * CC * CC, 128));
  ChainBwdParams p;
  p.N = N; p.has_k2 = has_k2;
  const char* tr = getenv("GLF_CHAIN_TRACE");
  p.trace = (tr && tr[0] == '1') ? 1 : 0;
  p.sfv = sfv; p.cvec = cvec; p.rv = rv; p.k1 = k1; p.k2 = k2; p.k3 = k3;
  p.bth = bth; p.bphi = bphi; p.bg = bg;
  p.Rb = Rb;
  p.dQa = dQa; p.dWp = dWp; p.dMn = dMn; p.dT = dT; p.EF = EF; p.evec = evec;
  p.dcv = dcv; p.dtv = dtv;
  cudaError_t e = cudaFuncSetAttribute(chain_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CH_SMEM);
  if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(chain_bwd)");
  chain_bwd_kernel<<<B, CH_THREADS, CH_SMEM, stream>>>(tmS, tmQ, tmW, tmWz, tmdQ, tmdWp, tmdM, tmdT, tmEF, tmR, p);
  if (p.trace) {
    static const char* names[] = {"start", "LDA", "MMAA", "LDB", "MMAB", "DRA", "LDC", "MMAC", "DRB", "LDD", "MMAD", "DRC", "LDE", "MMAE", "DRD", "LDF", "MMAF", "DRE", "LDH", "DRK0", "DRK1", "DRF", "end"};
    long long t[64];
    cudaStreamSynchronize(stream);
    cudaMemcpyFromSymbol(t, g_chain_trace, sizeof(t));
    fprintf(stderr, "chain_bwd trace (SM cycles since start, delta):");
    for (int i = 1; i <= 21; ++i) fprintf(stderr, " %s=%lld(+%lld)", names[i], t[i] - t[0], t[i] - t[i - 1]);
    fprintf(stderr, "\n");
  }
  return check_cuda(cudaGetLastError(), "chain_bwd launch");
}

}  // namespace glf
