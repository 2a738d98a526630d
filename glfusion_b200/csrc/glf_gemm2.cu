// glf_gemm2.cu — the big K-major products of the Gram form (U = X Q^T + c, dX = [dV | X][E' ; F] + e: M = tokens, N = 256)
// on CTA PAIRS: tcgen05.mma.cta_group::2.
//
// The single-CTA tile GEMM (glf_gemm.cu) is bound, for these shapes, by its epilogue and by the L2 -> SM operand bytes
// (profiles/r02_gemm_bound_probe.txt): a 256 x 128 CTA tile pulls (256 + 128) K elements per 32 K outputs.  Here a
// cluster of two CTAs owns a 256 x 256 tile: each CTA loads ITS 128 rows of A and ITS half (128 of 256 rows) of B, the
// leader issues one M = 256, N = 256 MMA per K step that reads both CTAs' shared memory and writes both CTAs' TMEM
// (128 lanes x 256 columns each, two accumulator stages), so the operand bytes per output drop by a third while every
// CTA keeps a double-buffered accumulator and the full 16-warp epilogue of a 128 x 256 tile.
//
//   warp 0      TMA producer (both CTAs): own A tile + own B half into a 5-stage ring (32 KB per stage); the bytes are
//               counted on the LEADER's full barrier (cp.async.bulk.tensor ... .cta_group::2)
//   warp 1      MMA issuer (leader only); tcgen05.commit multicasts to both CTAs' empty / accumulator-full barriers
//   warps 2-17  epilogue (both CTAs): tcgen05.ld -> bias -> bf16 staging -> bulk tensor stores (+ BatchNorm column
//               statistics, one partial row per 32-row sub-block); the last read of an accumulator stage arrives on the
//               LEADER's accumulator-empty barrier (count = both CTAs' epilogue warps)
#include "glf_internal.h"
#include "glf_ptx.cuh"

namespace glf {

namespace {

constexpr int BM = 128, BN2 = 256, BK = 64;
constexpr int G2_STAGES = 5;
constexpr int EPI_WARPS = 16;
constexpr int EPI_THREADS = EPI_WARPS * 32;
constexpr int G2_THREADS = 64 + EPI_THREADS;
constexpr uint32_t G2_A = BM * BK * 2;           // this CTA's 128 rows of A, one k-block
constexpr uint32_t G2_B = 128 * BK * 2;          // this CTA's 128 of the 256 B rows
constexpr uint32_t G2_STAGE = G2_A + G2_B;
constexpr uint32_t G2_RING = G2_STAGES * G2_STAGE;
constexpr uint32_t WARP_STG = 32 * 64, WARP_BIAS = 32 * 4;
// two staging tiles per epilogue warp: the bulk store of one chunk drains while the next chunk is packed
constexpr uint32_t G2_EPI = EPI_WARPS * (2 * WARP_STG + WARP_BIAS);
constexpr uint32_t G2_SMEM = G2_RING + G2_EPI + 256 + 512;
static_assert(G2_SMEM <= 232448, "shared memory budget");

struct Gemm2Params {
  int M, N, batch, kb_total, npairs;
  int pairA[6], pairB[6];
  int a_batched, b_batched;
  int tiles_m;             // 256-row pair tiles per batch entry
  int tiles_n;             // 256-column tiles (N / 256); the tile index runs n fastest
  int total;               // pair tiles
  const float* bias;
  long long bias_stride;
  float* colstats;         // [batch * tiles_m128 * 4][2][N]: one partial row per 32-row sub-block (or null),
  int tiles_m128;          //    the single-CTA kernel's table layout
  float alpha;
  const bf16* addend;      // optional bf16 [M, N] added before the store
  long long ld_add, stride_add;
  int split_k, kb_per_split;   // K slices per tile (fp32 atomic output only)
  float* Df;               // out_kind 2: fp32 output, red.global.add (split-K slices / batch-reduced products)
  long long ldd, strideD;
};

__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

template <bool A_MN, bool B_MN>
__global__ void __launch_bounds__(G2_THREADS, 1)
    gemm_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                     const __grid_constant__ CUtensorMap tmD, const Gemm2Params p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  if (smem_base - smem_u32(smem_raw) > 512u) __trap();
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  uint8_t* epi_smem = smem_gen + G2_RING;
  uint64_t* bar_mem = reinterpret_cast<uint64_t*>(smem_gen + G2_RING + G2_EPI);
  uint64_t* full_bar = bar_mem;             // [6]   (the leader's are the ones in use)
  uint64_t* empty_bar = bar_mem + 8;        // [6]
  uint64_t* tmem_full_bar = bar_mem + 16;   // [2]
  uint64_t* tmem_empty_bar = bar_mem + 18;  // [2]   (the leader's are the ones in use)
  uint32_t& tmem_holder = *reinterpret_cast<uint32_t*>(bar_mem + 20);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int cluster_id = blockIdx.x >> 1, nclusters = gridDim.x >> 1;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmD);
#pragma unroll
    for (int s = 0; s < G2_STAGES; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      mbar_init(smem_u32(&tmem_full_bar[s]), 1);
      mbar_init(smem_u32(&tmem_empty_bar[s]), 2 * EPI_WARPS);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc_cg2(smem_u32(&tmem_holder), 512);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();      // both CTAs' barriers are initialised, both TMEM allocations are visible
  tc_fence_after();
  const uint32_t tmem_base = tmem_holder;

  if (warp == 0) {
    // ------------------------------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int item = cluster_id; item < p.total * p.split_k; item += nclusters) {
        const int tile = item / p.split_k, ks = item - tile * p.split_k;
        const int nt = tile % p.tiles_n, bm = tile / p.tiles_n;
        const int b = bm / p.tiles_m, mt = bm - b * p.tiles_m;
        const int m0 = mt * 256 + static_cast<int>(rank) * BM, n0 = nt * BN2 + static_cast<int>(rank) * 128;
        const int ab = p.a_batched ? b : 0, bb = p.b_batched ? b : 0;
        const int kb0 = ks * p.kb_per_split;
        const int niter = (min(p.kb_total, kb0 + p.kb_per_split) - kb0) * p.npairs;
        for (int it = 0; it < niter; ++it) {
          const int pair = it % p.npairs;
          const int k0 = (kb0 + it / p.npairs) * BK;
          mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1u);
          if (leader) mbar_expect_tx(smem_u32(&full_bar[stage]), 2 * G2_STAGE);   // both CTAs' bytes
          const uint32_t fb = mapa_shared(smem_u32(&full_bar[stage]), 0);
          const uint32_t sa = smem_base + stage * G2_STAGE, sb = sa + G2_A;
          if (!A_MN) {
            tma_load_4d_cg2(&tmA, fb, sa, k0, m0, ab, p.pairA[pair]);
          } else {                 // MN-major A (token contractions): two [64 k][64 m] boxes, the image `mdesc` reads
            tma_load_4d_cg2(&tmA, fb, sa, m0, k0, ab, p.pairA[pair]);
            tma_load_4d_cg2(&tmA, fb, sa + 8192, m0 + 64, k0, ab, p.pairA[pair]);
          }
          if (!B_MN) {
            tma_load_4d_cg2(&tmB, fb, sb, k0, n0, bb, p.pairB[pair]);
          } else {
            tma_load_4d_cg2(&tmB, fb, sb, n0, k0, bb, p.pairB[pair]);
            tma_load_4d_cg2(&tmB, fb, sb + 8192, n0 + 64, k0, bb, p.pairB[pair]);
          }
          if (++stage == G2_STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------------------------------ MMA issuer (leader)
    if (leader && elect_one()) {
      constexpr uint32_t idesc = make_idesc_bf16(256, BN2, A_MN, B_MN);
      int stage = 0;
      uint32_t phase = 0;
      int local = 0;
      for (int item = cluster_id; item < p.total * p.split_k; item += nclusters, ++local) {
        const int kb0 = (item % p.split_k) * p.kb_per_split;
        const int niter = (min(p.kb_total, kb0 + p.kb_per_split) - kb0) * p.npairs;
        const int acc = local & 1;
        const uint32_t use = static_cast<uint32_t>(local >> 1);
        mbar_wait(smem_u32(&tmem_empty_bar[acc]), (use & 1u) ^ 1u);   // both CTAs' epilogues drained this stage
        tc_fence_after();
        const uint32_t tacc = tmem_base + acc * BN2;
        for (int it = 0; it < niter; ++it) {
          mbar_wait(smem_u32(&full_bar[stage]), phase);
          tc_fence_after();
          const uint32_t sa = smem_base + stage * G2_STAGE, sb = sa + G2_A;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint64_t ad = A_MN ? make_sdesc(sa + k * 2048, 8192, 1024) : make_sdesc(sa + k * 32, 16, 1024);
            const uint64_t bd = B_MN ? make_sdesc(sb + k * 2048, 8192, 1024) : make_sdesc(sb + k * 32, 16, 1024);
            umma_f16_cg2(tacc, ad, bd, idesc, (it | k) != 0 ? 1u : 0u);
          }
          umma_commit_cg2_mcast(smem_u32(&empty_bar[stage]), static_cast<uint16_t>(3));
          if (++stage == G2_STAGES) { stage = 0; phase ^= 1u; }
        }
        umma_commit_cg2_mcast(smem_u32(&tmem_full_bar[acc]), static_cast<uint16_t>(3));
      }
    }
  } else {
    // ------------------------------------------------------------------------------------------ epilogue
    const int ew = warp - 2, q = warp & 3, cc0 = ew >> 2;
    constexpr int NCHUNK = BN2 / 32;          // 8: warp (q, cc0) owns chunks cc0 and cc0 + 4
    uint8_t* wstg0 = epi_smem + ew * 2 * WARP_STG;
    float* wbias = reinterpret_cast<float*>(epi_smem + EPI_WARPS * 2 * WARP_STG + ew * WARP_BIAS);
    int nchunk = 0;
    const int sw_w = (lane >> 1) & 3;
    const int hl = lane & 15, half = lane >> 4;
    const uint32_t leader_empty0 = mapa_shared(smem_u32(&tmem_empty_bar[0]), 0);
    const uint32_t leader_empty1 = mapa_shared(smem_u32(&tmem_empty_bar[1]), 0);
    int local = 0;
    for (int item = cluster_id; item < p.total * p.split_k; item += nclusters, ++local) {
      const int tile = item / p.split_k;
      const int nt = tile % p.tiles_n, bm = tile / p.tiles_n;
      const int b = bm / p.tiles_m, mt = bm - b * p.tiles_m;
      const int m0 = mt * 256 + static_cast<int>(rank) * BM;
      const int acc = local & 1;
      const uint32_t use = static_cast<uint32_t>(local >> 1);
      const float* biasb = p.bias != nullptr ? p.bias + static_cast<long long>(b) * p.bias_stride : nullptr;
      const int rows_valid = min(32, p.M - (m0 + q * 32));
      // this warp's two bias slices are fetched BEFORE the wait for the accumulator: the global-load latency hides
      // behind the tile's MMAs
      float bpre0 = 0.f, bpre1 = 0.f;
      if (biasb != nullptr) {
        bpre0 = biasb[nt * BN2 + cc0 * 32 + lane];
        bpre1 = biasb[nt * BN2 + (cc0 + 4) * 32 + lane];
      }
      mbar_wait(smem_u32(&tmem_full_bar[acc]), use & 1u);
      tc_fence_after();
      const uint32_t taddr = tmem_base + acc * BN2 + (static_cast<uint32_t>(q * 32) << 16);
#pragma unroll 1
      for (int ci = 0; ci < 2; ++ci) {
        const int c = cc0 + 4 * ci;
        const int gc0 = nt * BN2 + c * 32;
        uint32_t v[32];
        tmem_ld_32x32(taddr + c * 32, v);
        if (biasb != nullptr) wbias[lane] = ci == 0 ? bpre0 : bpre1;
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (ci == 1 && lane == 0) mbar_arrive_cluster(acc == 0 ? leader_empty0 : leader_empty1);
        float2 f[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) f[j] = make_float2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
        if (p.alpha != 1.f) {
          const float2 al = make_float2(p.alpha, p.alpha);
#pragma unroll
          for (int j = 0; j < 16; ++j) f[j] = mul2(f[j], al);
        }
        if (biasb != nullptr) {
#pragma unroll
          for (int j = 0; j < 16; j += 2) {
            const float4 bv = *reinterpret_cast<const float4*>(wbias + 2 * j);
            f[j] = add2(f[j], make_float2(bv.x, bv.y));
            f[j + 1] = add2(f[j + 1], make_float2(bv.z, bv.w));
          }
        }
        if (p.Df != nullptr) {                                // fp32 atomic output: no staging, no bulk store
          if (lane < rows_valid) {
            float* dr = p.Df + static_cast<long long>(b) * p.strideD + static_cast<long long>(m0 + q * 32 + lane) * p.ldd + gc0;
#pragma unroll
            for (int j = 0; j < 16; j += 2) red_add_v4(dr + 2 * j, f[j].x, f[j].y, f[j + 1].x, f[j + 1].y);
          }
          __syncwarp();
          continue;
        }
        if (p.addend != nullptr && lane < rows_valid) {       // this lane's row: 32 bf16 = 64 contiguous bytes
          const uint4* ar = reinterpret_cast<const uint4*>(p.addend + static_cast<long long>(b) * p.stride_add +
                                                           static_cast<long long>(m0 + q * 32 + lane) * p.ld_add + gc0);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint4 a4 = __ldg(ar + j);
            f[4 * j] = add2(f[4 * j], unpack_bf16(a4.x));
            f[4 * j + 1] = add2(f[4 * j + 1], unpack_bf16(a4.y));
            f[4 * j + 2] = add2(f[4 * j + 2], unpack_bf16(a4.z));
            f[4 * j + 3] = add2(f[4 * j + 3], unpack_bf16(a4.w));
          }
        }
        uint8_t* wstg = wstg0 + (nchunk & 1) * WARP_STG;
        ++nchunk;
        if (lane == 0) tma_store_wait_read<1>();     // the bulk store issued TWO chunks ago has drained this tile
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint4 pk = make_uint4(pack_bf16(f[4 * j].x, f[4 * j].y), pack_bf16(f[4 * j + 1].x, f[4 * j + 1].y),
                                      pack_bf16(f[4 * j + 2].x, f[4 * j + 2].y),
                                      pack_bf16(f[4 * j + 3].x, f[4 * j + 3].y));
          *reinterpret_cast<uint4*>(wstg + lane * 64 + ((j ^ sw_w) << 4)) = pk;
        }
        __syncwarp();
        if (p.colstats != nullptr) {
          // sums of the stored (bf16-rounded) values over the sub-block's valid rows, on column pairs (see glf_gemm.cu)
          float2 sa2 = make_float2(0.f, 0.f), sq2 = make_float2(0.f, 0.f);
          const uint8_t* src = wstg + half * 16 * 64 + (hl & 3) * 4;
          if (rows_valid >= 32) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float2 x = unpack_bf16(
                  *reinterpret_cast<const uint32_t*>(src + i * 64 + (((hl >> 2) ^ ((i >> 1) & 3)) << 4)));
              sa2 = add2(sa2, x);
              sq2 = fma2(x, x, sq2);
            }
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              if (half * 16 + i < rows_valid) {
                const float2 x = unpack_bf16(
                    *reinterpret_cast<const uint32_t*>(src + i * 64 + (((hl >> 2) ^ ((i >> 1) & 3)) << 4)));
                sa2 = add2(sa2, x);
                sq2 = fma2(x, x, sq2);
              }
            }
          }
          sa2.x += __shfl_xor_sync(0xffffffffu, sa2.x, 16);
          sa2.y += __shfl_xor_sync(0xffffffffu, sa2.y, 16);
          sq2.x += __shfl_xor_sync(0xffffffffu, sq2.x, 16);
          sq2.y += __shfl_xor_sync(0xffffffffu, sq2.y, 16);
          if (half == 0 && m0 < p.M) {                         // (a 128-row half entirely beyond M has no table rows)
            float* cs = p.colstats + ((static_cast<long long>(b) * p.tiles_m128 + (m0 >> 7)) * 4 + q) * 2 * p.N;
            *reinterpret_cast<float2*>(cs + gc0 + 2 * hl) = sa2;
            *reinterpret_cast<float2*>(cs + p.N + gc0 + 2 * hl) = sq2;
          }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_3d(&tmD, smem_u32(wstg), gc0, m0 + q * 32, b);    // rows / columns beyond M / N are clipped
          tma_store_commit();
        }
      }
    }
    if (lane == 0) tma_store_wait_all<0>();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();      // no CTA leaves (or frees its TMEM) while the pair's MMAs / remote arrivals may be in flight
  if (warp == 1) tmem_dealloc_cg2(tmem_base, 512);
}

template <bool A_MN, bool B_MN>
int launch_pair(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmD, const Gemm2Params& p, int grid,
                cudaStream_t stream) {
  auto kern = gemm_pair_kernel<A_MN, B_MN>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, G2_SMEM);
  if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(gemm_pair)");
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(G2_THREADS);
  cfg.dynamicSmemBytes = G2_SMEM;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return check_cuda(cudaLaunchKernelEx(&cfg, kern, tmA, tmB, tmD, p), "gemm_pair launch");
}

}  // namespace

bool gemm_pair_applicable(const GemmArgs& a, int num_sms) {
  if (a.N % BN2 != 0 || a.M < 1024 || a.out_kind == 1 || a.rowsum != nullptr) return false;
  if (a.npairs > 6 || num_sms < 2) return false;
  if (a.out_kind == 0 && (a.split_k > 1 || a.strideD % 8 != 0)) return false;
  if (a.out_kind == 2 && (a.bias != nullptr || a.addend != nullptr || a.colstats != nullptr || a.ldd % 4 != 0 ||
                          a.strideD % 4 != 0 || (reinterpret_cast<uintptr_t>(a.D) & 15) != 0))
    return false;
  // MN-major A is the token contraction of the token-space path (K = tokens): worth a pair only when tensor-bound
  if (a.A.mn_major && (a.M % 128 != 0 || static_cast<long long>(a.M) * a.N < 1024 * 1024)) return false;
  if (a.K % BK != 0 && !(a.A.mn_major && a.B.mn_major)) return false;   // (a K tail is zero-filled by TMA for MN-major operands)
  if (a.addend != nullptr && (a.ld_add % 8 != 0 || a.stride_add % 8 != 0 || (reinterpret_cast<uintptr_t>(a.addend) & 15) != 0))
    return false;
  // measured at K = 256: with the column statistics in the epilogue the single-CTA tile is faster (HBM-bound shape)
  if (a.colstats != nullptr && a.N == BN2) return false;
  // several column tiles (the C = 2048 products): per-sub-block partial rows; worth it once the product is tensor-bound
  if (a.colstats != nullptr && a.K < 1024) return false;
  const long long tiles = static_cast<long long>((a.M + 255) / 256) * a.batch * (a.N / BN2) * (a.split_k > 1 ? a.split_k : 1);
  const int grid = (num_sms / 2) * 2;
  if (tiles < grid / 2) return false;            // not enough pair tiles to fill the machine
  return true;
}

int gemm_pair(const GemmArgs& a, int num_sms, cudaStream_t stream) {
  int nlimbsA = 1, nlimbsB = 1;
  for (int i = 0; i < a.npairs; ++i) {
    nlimbsA = a.pairA[i] + 1 > nlimbsA ? a.pairA[i] + 1 : nlimbsA;
    nlimbsB = a.pairB[i] + 1 > nlimbsB ? a.pairB[i] + 1 : nlimbsB;
  }
  CUtensorMap tmA, tmB, tmD;
  int rc = make_operand_tmap(&tmA, a.A, a.A.rows > 0 ? a.A.rows : a.M, a.K, a.batch, nlimbsA, BM);
  if (rc) return rc;
  rc = make_operand_tmap(&tmB, a.B, a.B.rows > 0 ? a.B.rows : a.N, a.K, a.batch, nlimbsB, 128);
  if (rc) return rc;
  if (a.out_kind == 0) {
    rc = make_output_tmap(&tmD, a.D, a.M, a.N, a.batch, a.ldd, a.strideD);
    if (rc) return rc;
  } else {
    tmD = tmA;     // unused by the fp32 atomic epilogue
  }
  Gemm2Params p;
  p.M = a.M; p.N = a.N; p.batch = a.batch;
  p.kb_total = (a.K + BK - 1) / BK;
  {
    const int sk = a.split_k < 1 ? 1 : a.split_k;
    p.kb_per_split = (p.kb_total + sk - 1) / sk;
    p.split_k = (p.kb_total + p.kb_per_split - 1) / p.kb_per_split;
  }
  p.Df = a.out_kind == 2 ? reinterpret_cast<float*>(a.D) : nullptr;
  p.ldd = a.ldd;
  p.strideD = a.strideD;
  p.npairs = a.npairs;
  for (int i = 0; i < 6; ++i) { p.pairA[i] = a.pairA[i]; p.pairB[i] = a.pairB[i]; }
  p.a_batched = a.A.batch_stride != 0;
  p.b_batched = a.B.batch_stride != 0;
  p.tiles_m = (a.M + 255) / 256;
  p.tiles_n = a.N / BN2;
  p.total = p.tiles_m * a.batch * p.tiles_n;
  p.bias = a.bias;
  p.bias_stride = a.bias != nullptr ? a.bias_stride : 0;
  p.colstats = a.colstats;
  p.tiles_m128 = gemm_tiles_m(a.M);
  p.alpha = a.alpha;
  p.addend = a.addend;
  p.ld_add = a.ld_add;
  p.stride_add = a.stride_add;
  const int grid = (num_sms / 2) * 2;
  if (a.colstats_rows != nullptr) *a.colstats_rows = a.colstats == nullptr ? 0 : a.batch * p.tiles_m128 * 4;
  if (a.A.mn_major)
    return a.B.mn_major ? launch_pair<true, true>(tmA, tmB, tmD, p, grid, stream)
                        : launch_pair<true, false>(tmA, tmB, tmD, p, grid, stream);
  return a.B.mn_major ? launch_pair<false, true>(tmA, tmB, tmD, p, grid, stream)
                      : launch_pair<false, false>(tmA, tmB, tmD, p, grid, stream);
}

}  // namespace glf
