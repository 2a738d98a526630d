// glf_gemm3.cu — U = X Q^T + c of the Gram form (M = tokens, N = 256, K = 256, one [256 x 256] B operand PER SEQUENCE)
// with the B operand RESIDENT in shared memory.
//
// The tile GEMMs (glf_gemm.cu / glf_gemm2.cu) re-fetch B for every output tile: for U that is 128 KB of B per 64 KB of A,
// and the kernel ends up bound by the L2 -> SM fabric (profiles/r02_gemm_bound_probe.txt: 602 MB of operand bytes per
// launch at ~10 TB/s = 60 us with no epilogue at all, for 205 MB of unique input).  All 24.5 row tiles of a sequence
// multiply the SAME Q, so here every CTA owns a CONTIGUOUS range of 128-row tiles (21 - 22 of them: at most two
// sequences), keeps that sequence's Q (128 KB, four [256 n][64 k] SWIZZLE_128B tiles) in shared memory and streams only
// A through a 4-stage ring: operand bytes per launch drop to A once + Q once per CTA and sequence, i.e. HBM-bound.
//
//   warp 0      TMA producer: Q when the sequence changes (after the MMAs on the previous Q have retired), A k-blocks
//   warp 1      MMA issuer: M = 128, N = 256, K = 16 tcgen05.mma, two TMEM accumulator stages of 256 columns
//   warps 2-17  epilogue: tcgen05.ld -> per-sequence bias -> bf16 staging -> bulk tensor store (+ BatchNorm column
//               statistics of the stored values as per-CTA running sums, one partial row per CTA, fixed order)
#include "glf_internal.h"
#include "glf_ptx.cuh"

namespace glf {

namespace {

constexpr int BM = 128, BN3 = 256, BK = 64;
constexpr int G3_STAGES = 4;
constexpr int G3_KB_MAX = 4;                          // K <= 256
constexpr int EPI_WARPS = 16;
constexpr int EPI_THREADS = EPI_WARPS * 32;
constexpr int G3_THREADS = 64 + EPI_THREADS;
constexpr uint32_t G3_A = BM * BK * 2;                // 16 KB per k-block
constexpr uint32_t G3_BT = BN3 * BK * 2;              // 32 KB per k-block of the resident operand
constexpr uint32_t G3_B = G3_KB_MAX * G3_BT;          // 128 KB
constexpr uint32_t G3_RING = G3_STAGES * G3_A;        // 64 KB = one full A tile in flight
constexpr uint32_t WARP_STG = 32 * 64, WARP_BIAS = 32 * 4;
constexpr uint32_t G3_EPI = EPI_WARPS * (WARP_STG + WARP_BIAS);
constexpr uint32_t G3_SMEM = G3_B + G3_RING + G3_EPI + 256 + 512;
static_assert(G3_SMEM <= 232448, "shared memory budget");

struct Gemm3Params {
  int M, N, batch, kb_total;
  int a_batched, b_batched;
  int tiles_m;             // 128-row tiles per batch entry
  int total;               // tiles
  const float* bias;
  long long bias_stride;
  float* colstats;         // [gridDim.x][2][N] per-CTA running sums (or null)
  float alpha;
};

__global__ void __launch_bounds__(G3_THREADS, 1)
    gemm_bres_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                     const __grid_constant__ CUtensorMap tmD, const Gemm3Params p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  if (smem_base - smem_u32(smem_raw) > 512u) __trap();
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t sB = smem_base, sRing = smem_base + G3_B;
  uint8_t* epi_smem = smem_gen + G3_B + G3_RING;
  uint64_t* bar_mem = reinterpret_cast<uint64_t*>(smem_gen + G3_B + G3_RING + G3_EPI);
  uint64_t* full_bar = bar_mem;             // [4]
  uint64_t* empty_bar = bar_mem + 4;        // [4]
  uint64_t* tmem_full_bar = bar_mem + 8;    // [2]
  uint64_t* tmem_empty_bar = bar_mem + 10;  // [2]
  uint64_t* b_full_bar = bar_mem + 12;      // resident operand landed
  uint64_t* b_empty_bar = bar_mem + 13;     // every MMA on the resident operand has retired
  uint32_t& tmem_holder = *reinterpret_cast<uint32_t*>(bar_mem + 14);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // contiguous tile range of this CTA
  const int t_begin = static_cast<int>(static_cast<long long>(p.total) * blockIdx.x / gridDim.x);
  const int t_end = static_cast<int>(static_cast<long long>(p.total) * (blockIdx.x + 1) / gridDim.x);

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmD);
#pragma unroll
    for (int s = 0; s < G3_STAGES; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      mbar_init(smem_u32(&tmem_full_bar[s]), 1);
      mbar_init(smem_u32(&tmem_empty_bar[s]), EPI_WARPS);
    }
    mbar_init(smem_u32(b_full_bar), 1);
    mbar_init(smem_u32(b_empty_bar), 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_holder), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_holder;

  if (warp == 0) {
    // ------------------------------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      int cur_b = -1;
      uint32_t b_loads = 0;
      for (int tile = t_begin; tile < t_end; ++tile) {
        const int b = tile / p.tiles_m, mt = tile - b * p.tiles_m;
        if (b != cur_b) {
          // the MMAs that read the previous sequence's operand must have retired before it is overwritten
          if (b_loads > 0) mbar_wait(smem_u32(b_empty_bar), (b_loads - 1) & 1u);
          mbar_expect_tx(smem_u32(b_full_bar), static_cast<uint32_t>(p.kb_total) * G3_BT);
          for (int kb = 0; kb < p.kb_total; ++kb) {
            tma_load_4d(&tmB, smem_u32(b_full_bar), sB + kb * G3_BT, kb * BK, 0, p.b_batched ? b : 0, 0);
            tma_load_4d(&tmB, smem_u32(b_full_bar), sB + kb * G3_BT + G3_BT / 2, kb * BK, 128, p.b_batched ? b : 0, 0);
          }
          cur_b = b;
          ++b_loads;
        }
        for (int kb = 0; kb < p.kb_total; ++kb) {
          mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1u);
          mbar_expect_tx(smem_u32(&full_bar[stage]), G3_A);
          tma_load_4d(&tmA, smem_u32(&full_bar[stage]), sRing + stage * G3_A, kb * BK, mt * BM, p.a_batched ? b : 0, 0);
          if (++stage == G3_STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------------------------------ MMA issuer
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc_bf16(BM, BN3, false, false);
      int stage = 0;
      uint32_t phase = 0;
      int local = 0, cur_b = -1;
      uint32_t b_uses = 0;
      for (int tile = t_begin; tile < t_end; ++tile, ++local) {
        const int b = tile / p.tiles_m;
        if (b != cur_b) {
          mbar_wait(smem_u32(b_full_bar), b_uses & 1u);
          tc_fence_after();
          cur_b = b;
          ++b_uses;
        }
        const int acc = local & 1;
        const uint32_t use = static_cast<uint32_t>(local >> 1);
        mbar_wait(smem_u32(&tmem_empty_bar[acc]), (use & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t tacc = tmem_base + acc * BN3;
        for (int kb = 0; kb < p.kb_total; ++kb) {
          mbar_wait(smem_u32(&full_bar[stage]), phase);
          tc_fence_after();
          const uint32_t sa = sRing + stage * G3_A, sb = sB + kb * G3_BT;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint64_t ad = make_sdesc(sa + k * 32, 16, 1024);
            const uint64_t bd = make_sdesc(sb + k * 32, 16, 1024);
            umma_f16(tacc, ad, bd, idesc, (kb | k) != 0 ? 1u : 0u);
          }
          umma_commit(smem_u32(&empty_bar[stage]));
          if (++stage == G3_STAGES) { stage = 0; phase ^= 1u; }
        }
        umma_commit(smem_u32(&tmem_full_bar[acc]));
        // last tile on this sequence's operand: tell the producer when these MMAs have retired
        const bool last_on_b = tile + 1 >= t_end || (tile + 1) / p.tiles_m != b;
        if (last_on_b) umma_commit(smem_u32(b_empty_bar));
      }
    }
  } else {
    // ------------------------------------------------------------------------------------------ epilogue
    const int ew = warp - 2, q = warp & 3, cc0 = ew >> 2;      // warp (q, cc0) owns 32-column chunks cc0 and cc0 + 4
    uint8_t* wstg = epi_smem + ew * WARP_STG;
    float* wbias = reinterpret_cast<float*>(epi_smem + EPI_WARPS * WARP_STG + ew * WARP_BIAS);
    const int sw_w = (lane >> 1) & 3;
    const int hl = lane & 15, half = lane >> 4;
    float2 cs1[2], cs2[2];
    cs1[0] = cs1[1] = cs2[0] = cs2[1] = make_float2(0.f, 0.f);
    int local = 0;
    for (int tile = t_begin; tile < t_end; ++tile, ++local) {
      const int b = tile / p.tiles_m, mt = tile - b * p.tiles_m;
      const int m0 = mt * BM;
      const int acc = local & 1;
      const uint32_t use = static_cast<uint32_t>(local >> 1);
      const float* biasb = p.bias != nullptr ? p.bias + static_cast<long long>(b) * p.bias_stride : nullptr;
      const int rows_valid = min(32, p.M - (m0 + q * 32));
      float bpre0 = 0.f, bpre1 = 0.f;              // fetched before the accumulator wait
      if (biasb != nullptr) {
        bpre0 = biasb[cc0 * 32 + lane];
        bpre1 = biasb[(cc0 + 4) * 32 + lane];
      }
      mbar_wait(smem_u32(&tmem_full_bar[acc]), use & 1u);
      tc_fence_after();
      const uint32_t taddr = tmem_base + acc * BN3 + (static_cast<uint32_t>(q * 32) << 16);
#pragma unroll 1
      for (int ci = 0; ci < 2; ++ci) {
        const int c = cc0 + 4 * ci;
        const int gc0 = c * 32;
        uint32_t v[32];
        tmem_ld_32x32(taddr + c * 32, v);
        if (biasb != nullptr) wbias[lane] = ci == 0 ? bpre0 : bpre1;
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (ci == 1 && lane == 0) mbar_arrive(smem_u32(&tmem_empty_bar[acc]));
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
        if (lane == 0) tma_store_wait_read<0>();     // the previous chunk's bulk store has drained the staging tile
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
          // sums of the stored (bf16-rounded) values over the sub-block's valid rows, on column pairs
          float2 sa2 = make_float2(0.f, 0.f), sq2 = make_float2(0.f, 0.f);
          const uint8_t* src = wstg + half * 16 * 64 + (hl & 3) * 4;
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            if (rows_valid >= 32 || half * 16 + i < rows_valid) {
              const float2 x = unpack_bf16(
                  *reinterpret_cast<const uint32_t*>(src + i * 64 + (((hl >> 2) ^ ((i >> 1) & 3)) << 4)));
              sa2 = add2(sa2, x);
              sq2 = fma2(x, x, sq2);
            }
          }
          sa2.x += __shfl_xor_sync(0xffffffffu, sa2.x, 16);
          sa2.y += __shfl_xor_sync(0xffffffffu, sa2.y, 16);
          sq2.x += __shfl_xor_sync(0xffffffffu, sq2.x, 16);
          sq2.y += __shfl_xor_sync(0xffffffffu, sq2.y, 16);
          cs1[ci] = add2(cs1[ci], sa2);
          cs2[ci] = add2(cs2[ci], sq2);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_3d(&tmD, smem_u32(wstg), gc0, m0 + q * 32, b);    // rows beyond M are clipped
          tma_store_commit();
        }
      }
    }
    if (lane == 0) tma_store_wait_all<0>();
    if (p.colstats != nullptr) {
      // ONE partial row per CTA: the four warps that share a column chunk (one per 32-row quarter) combine their
      // running sums through the idle staging tiles, in a fixed order
      __syncwarp();
      float2* xs = reinterpret_cast<float2*>(wstg);            // [slot][sum | sum of squares][16 column pairs]
      if (half == 0) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          xs[(2 * i) * 16 + hl] = cs1[i];
          xs[(2 * i + 1) * 16 + hl] = cs2[i];
        }
      }
      named_bar_sync(1, EPI_THREADS);
      if ((ew & 3) == 0 && half == 0) {
        float* cs = p.colstats + static_cast<long long>(blockIdx.x) * 2 * p.N;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int col = (cc0 + 4 * i) * 32 + 2 * hl;
          float2 t1 = make_float2(0.f, 0.f), t2 = make_float2(0.f, 0.f);
#pragma unroll
          for (int w4 = 0; w4 < 4; ++w4) {
            const float2* o = reinterpret_cast<const float2*>(wstg + w4 * WARP_STG);
            t1 = add2(t1, o[(2 * i) * 16 + hl]);
            t2 = add2(t2, o[(2 * i + 1) * 16 + hl]);
          }
          *reinterpret_cast<float2*>(cs + col) = t1;
          *reinterpret_cast<float2*>(cs + p.N + col) = t2;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

}  // namespace

bool gemm_bres_applicable(const GemmArgs& a, int num_sms) {
  if (a.A.mn_major || a.B.mn_major || a.N != BN3 || a.K % BK != 0 || a.K > G3_KB_MAX * BK) return false;
  if (a.out_kind != 0 || a.addend != nullptr || a.rowsum != nullptr || a.split_k > 1 || a.npairs != 1) return false;
  if (a.A.limb_stride != 0 || a.B.limb_stride != 0 || a.strideD % 8 != 0) return false;
  // worth it when many row tiles share one B operand
  const long long tiles_m = (a.M + BM - 1) / BM;
  if (tiles_m < 8 || tiles_m * a.batch < 2LL * num_sms) return false;
  if (a.colstats != nullptr && num_sms > static_cast<long long>(a.batch) * tiles_m * 4) return false;
  return true;
}

int gemm_bres(const GemmArgs& a, int num_sms, cudaStream_t stream) {
  CUtensorMap tmA, tmB, tmD;
  int rc = make_operand_tmap(&tmA, a.A, a.A.rows > 0 ? a.A.rows : a.M, a.K, a.batch, 1, BM);
  if (rc) return rc;
  rc = make_operand_tmap(&tmB, a.B, a.B.rows > 0 ? a.B.rows : a.N, a.K, a.batch, 1, 128);
  if (rc) return rc;
  rc = make_output_tmap(&tmD, a.D, a.M, a.N, a.batch, a.ldd, a.strideD);
  if (rc) return rc;
  Gemm3Params p;
  p.M = a.M; p.N = a.N; p.batch = a.batch;
  p.kb_total = a.K / BK;
  p.a_batched = a.A.batch_stride != 0;
  p.b_batched = a.B.batch_stride != 0;
  p.tiles_m = (a.M + BM - 1) / BM;
  p.total = p.tiles_m * a.batch;
  p.bias = a.bias;
  p.bias_stride = a.bias != nullptr ? a.bias_stride : 0;
  p.colstats = a.colstats;
  p.alpha = a.alpha;
  const int grid = num_sms < p.total ? num_sms : p.total;
  if (a.colstats_rows != nullptr) *a.colstats_rows = a.colstats != nullptr ? grid : 0;
  cudaError_t e = cudaFuncSetAttribute(gemm_bres_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, G3_SMEM);
  if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(gemm_bres)");
  gemm_bres_kernel<<<grid, G3_THREADS, G3_SMEM, stream>>>(tmA, tmB, tmD, p);
  return check_cuda(cudaGetLastError(), "gemm_bres launch");
}

}  // namespace glf
