// glf_gemm.cu — warp-specialised tcgen05 / TMEM / TMA GEMM for sm_100a.
//
//   D[b] = alpha * sum_p A_p[b] * B_p[b]^T (+ bias) (+ addend)          A: M x K, B: N x K, bf16 in, fp32 accumulate
//
// Persistent kernel, one CTA per SM; each CTA loops over 128 x BN output tiles (one batch entry / K split each):
//   warp 0      TMA producer  : cp.async.bulk.tensor 4-D loads (inner, rows, batch, limb) into a STAGES-deep ring,
//                               SWIZZLE_128B, completion on mbarriers
//   warp 1      MMA issuer    : allocates TMEM (two accumulator stages), one elected lane issues tcgen05.mma
//                               (M=128, N=BN, K=16) x 4 per stage; tcgen05.commit releases the smem slot / publishes
//                               the accumulator, so tile i+1 is computed while tile i is still in its epilogue
//   warps 2..17 epilogue      : 16 independent warps (no block barriers); each tcgen05.ld's its 32x32 sub-block of the
//                               fp32 accumulator, applies alpha/bias, then either fp32 store / fp32 red.add (split-K)
//                               from registers, or a warp-private swizzled smem transpose -> 64-byte row-segment
//                               stores (+ residual addend) and a per-sub-block column-statistics partial (sum, sum of
//                               squares) for the BatchNorm that follows W_z (ours.py:908).
// Operands may be K-major ([rows, K]) or MN-major ([K, rows]); the latter is how the token-contraction products
// (Phi^T G, dU^T Theta, dP^T X) read token-major activations without any transposed copy.
#include <mutex>

#include "glf_internal.h"
#include "glf_ptx.cuh"

namespace glf {

namespace {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int EPI_WARPS = 16;                 // 4 per SM sub-partition: the epilogue is a latency chain, it needs TLP
constexpr int EPI_THREADS = EPI_WARPS * 32;
constexpr int GEMM_THREADS = 64 + EPI_THREADS;  // warp 0 TMA, warp 1 MMA, warps 2..17 epilogue

struct GemmKParams {
  int M, N, K, batch;
  int kb_total, kb_per_split, split_k;
  int npairs;
  int pairA[6], pairB[6];
  int a_batched, b_batched;
  float alpha;
  const float* bias;
  int out_kind;
  void* D;
  long long ldd, strideD;
  const bf16* addend;
  long long ld_add, stride_add;
  float* colstats;
  unsigned mg_mn, mg_n, mg_sk;   // multiply-high magics for / tiles_mn, / tiles_n, / split_k
  int cs_accum;   // 1: column statistics accumulated per CTA over all its tiles (table rows = gridDim.x)
  int tiles_m, tiles_n;
  int step_n, step_m, step_z;    // (n-tile, m-tile, batch*split) advance per persistent-loop step of gridDim.x tiles
  int tma_store;                 // 1: bf16 output tiles leave through cp.async.bulk.tensor stores (tmD), no addend
  long long bias_stride;         // elements between the bias vectors of consecutive batch entries (0 = shared)
  float* rowsum;                 // optional [batch][M] fp32: sum over K of the A operand's row (BN <= 128, npairs == 1)
  long long rowsum_stride;
};

// MT = 128-row accumulators per CTA tile: MT = 2 computes a 256 x BN super-tile, so each k-block of the B operand is
// loaded once per 256 output rows instead of once per 128 (the big K-major products at C = 256 are bound by L2 -> SM
// traffic, not by HBM or the tensor pipe; profiles/r01_gram_gemm_ncu_brief.txt)
template <int BN, int MT = 1>
struct GemmCfg {
  // persistent kernel, one CTA per SM: ring + separate epilogue staging must fit in 227 KB
  // MT = 2: every spare byte goes to the ring (the big K-major products are bound by bytes in flight per SM: with
  // three 48 KB stages the ring turns over once per HBM round trip, ~76 GB/s per SM; profiles/r02_gemm_bound_probe.txt)
  static constexpr int STAGES = (MT == 2) ? 4 : ((BN == 256) ? 3 : ((BN == 128) ? 5 : 6));
  static constexpr uint32_t A_TILE = BM * BK * 2;
  static constexpr uint32_t A_BYTES = MT * A_TILE;
  static constexpr uint32_t B_BYTES = BN * BK * 2;
  static constexpr uint32_t STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr uint32_t RING_BYTES = STAGES * STAGE_BYTES;
  static constexpr uint32_t WARP_STG = 32 * 64;     // warp-private 32 rows x 32 bf16, XOR-swizzled 16-byte chunks
  static constexpr uint32_t WARP_BIAS = 32 * 4;     // warp-private bias slice of the current 32-column chunk
  // MT = 2 runs without the CTA-wide bias copy and the ones tile: those bytes go to the ring
  static constexpr uint32_t BIAS_ALL = (MT == 2) ? 0 : 4096 * 4;   // the whole bias vector (N <= 4096) is staged once per CTA
  static constexpr uint32_t EPI_BYTES = EPI_WARPS * (WARP_STG + WARP_BIAS) + BIAS_ALL;
  // all-ones K-major B tile [16 rows][64 k] for the row-sum side product (RING_BYTES and EPI_BYTES are multiples of
  // 1024, so it sits on a swizzle-atom boundary)
  static constexpr uint32_t ONES_BYTES = (MT == 2) ? 0 : 2048;
  static constexpr uint32_t BAR_BYTES = 256;        // mbarriers + TMEM address, after the ones tile
  static constexpr uint32_t SLACK = (MT == 2) ? 512 : 1024;   // alignment slack of the dynamic shared-memory base
  static constexpr uint32_t SMEM_BYTES = RING_BYTES + EPI_BYTES + ONES_BYTES + BAR_BYTES + SLACK;
  // two accumulator stages (+ two 16-column row-sum accumulators at column 2 BN when BN <= 128)
  static constexpr uint32_t TMEM_COLS = (BN == 64) ? 256 : 512;
  static constexpr uint32_t ACC_COLS = MT * BN;     // TMEM columns of one accumulator stage
  static constexpr int NACC = (2 * ACC_COLS <= TMEM_COLS) ? 2 : 1;   // accumulator stages
  static constexpr uint32_t RS_COL = 2 * BN;        // (MT == 1 only)
  static_assert(MT == 1 || (MT == 2 && BN == 128), "MT = 2 is instantiated for BN = 128");
  static_assert(NACC * ACC_COLS <= TMEM_COLS, "TMEM budget of the accumulator stages");
  static_assert(EPI_BYTES % 1024 == 0 && RING_BYTES % 1024 == 0, "ones tile alignment");
  static_assert(SMEM_BYTES <= 232448, "shared memory budget");
  static_assert(TMEM_COLS <= 512, "TMEM budget");
};

// n / d for a runtime-uniform d with magic = floor(2^32 / d): the estimate is q or q-1 for every n < 2^32, one
// correction step makes it exact (d == 1 is special-cased: its magic does not fit 32 bits)
__device__ __forceinline__ void fastdivmod(int n, int d, unsigned magic, int& q, int& r) {
  q = static_cast<int>(__umulhi(static_cast<unsigned>(n), magic));
  r = n - q * d;
  if (r >= d) { ++q; r -= d; }
  if (d == 1) { q = n; r = 0; }
}

__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// Persistent: CTA c processes tiles c, c + gridDim.x, ... ; tile index runs n-tile fastest, then m-tile, then
// (batch, k-split), so the CTAs that are resident together share A slabs through L2.
template <bool A_MN, bool B_MN, int BN, int MT = 1>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
    gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                const __grid_constant__ CUtensorMap tmD, const GemmKParams p) {
  using Cfg = GemmCfg<BN, MT>;
  static_assert(MT == 1 || !A_MN, "MT = 2 takes a K-major A operand");
  constexpr int BMT = BM * MT;                 // output rows of one CTA tile
  constexpr int STAGES = Cfg::STAGES;
  constexpr int NACC = Cfg::NACC;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  if (smem_base - smem_u32(smem_raw) > Cfg::SLACK) __trap();   // the carve-up below would overrun the allocation
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  uint8_t* epi_smem = smem_gen + Cfg::RING_BYTES;
  uint64_t* bar_mem = reinterpret_cast<uint64_t*>(smem_gen + Cfg::RING_BYTES + Cfg::EPI_BYTES + Cfg::ONES_BYTES);
  uint64_t* full_bar = bar_mem;                    // [STAGES]
  uint64_t* empty_bar = bar_mem + 8;               // [STAGES]
  uint64_t* tmem_full_bar = bar_mem + 16;          // [2]
  uint64_t* tmem_empty_bar = bar_mem + 18;         // [2]
  uint32_t& tmem_holder = *reinterpret_cast<uint32_t*>(bar_mem + 20);
  static_assert(STAGES <= 8, "barrier carve-up");

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int tiles_mn = p.tiles_m * p.tiles_n;
  const int total_tiles = tiles_mn * p.batch * p.split_k;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
#pragma unroll
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      mbar_init(smem_u32(&tmem_full_bar[s]), 1);
      mbar_init(smem_u32(&tmem_empty_bar[s]), EPI_WARPS);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_holder), Cfg::TMEM_COLS);
  const uint32_t ones_smem = smem_base + Cfg::RING_BYTES + Cfg::EPI_BYTES;
  if (p.rowsum != nullptr) {
    // bf16 1.0 everywhere: the swizzle pattern is irrelevant for a constant tile
    uint32_t* ones = reinterpret_cast<uint32_t*>(smem_gen + Cfg::RING_BYTES + Cfg::EPI_BYTES);
    for (int i = threadIdx.x; i < static_cast<int>(Cfg::ONES_BYTES / 4); i += GEMM_THREADS) ones[i] = 0x3F803F80u;
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_holder;

  if (warp == 0) {
    // ------------------------------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        int z, mn, mt, nt, b, split;
        fastdivmod(tile, tiles_mn, p.mg_mn, z, mn);
        fastdivmod(mn, p.tiles_n, p.mg_n, mt, nt);
        fastdivmod(z, p.split_k, p.mg_sk, b, split);
        const int m0 = mt * BMT, n0 = nt * BN;
        const int ab = p.a_batched ? b : 0, bb = p.b_batched ? b : 0;
        const int kb0 = split * p.kb_per_split;
        const int niter = (min(p.kb_total, kb0 + p.kb_per_split) - kb0) * p.npairs;
        for (int it = 0; it < niter; ++it) {
          const int pair = it % p.npairs;
          const int k0 = (kb0 + it / p.npairs) * BK;
          const uint32_t fb = smem_u32(&full_bar[stage]);
          mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1u);
          mbar_expect_tx(fb, Cfg::STAGE_BYTES);
          const uint32_t sa = smem_base + stage * Cfg::STAGE_BYTES;
          const uint32_t sb = sa + Cfg::A_BYTES;
          if (!A_MN) {
#pragma unroll
            for (int j = 0; j < MT; ++j) tma_load_4d(&tmA, fb, sa + j * Cfg::A_TILE, k0, m0 + j * BM, ab, p.pairA[pair]);
          } else {
            tma_load_4d(&tmA, fb, sa, m0, k0, ab, p.pairA[pair]);
            tma_load_4d(&tmA, fb, sa + 8192, m0 + 64, k0, ab, p.pairA[pair]);
          }
          if (!B_MN) {
            tma_load_4d(&tmB, fb, sb, k0, n0, bb, p.pairB[pair]);
          } else {
#pragma unroll
            for (int j = 0; j < BN / 64; ++j)
              tma_load_4d(&tmB, fb, sb + j * 8192, n0 + j * 64, k0, bb, p.pairB[pair]);
          }
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------------------------------ MMA issuer
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc_bf16(BM, BN, A_MN, B_MN);
      constexpr uint32_t idesc_rs = make_idesc_bf16(BM, 16, A_MN, false);
      int stage = 0;
      uint32_t phase = 0;
      int local = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++local) {
        int z, mn, b, split, mt_, nt_;
        fastdivmod(tile, tiles_mn, p.mg_mn, z, mn);
        fastdivmod(z, p.split_k, p.mg_sk, b, split);
        fastdivmod(mn, p.tiles_n, p.mg_n, mt_, nt_);
        const bool rs = MT == 1 && BN <= 128 && p.rowsum != nullptr && nt_ == 0;   // row sums ride along with the first n-tile
        const int kb0 = split * p.kb_per_split;
        const int niter = (min(p.kb_total, kb0 + p.kb_per_split) - kb0) * p.npairs;
        const int acc = local % NACC;
        const uint32_t use = static_cast<uint32_t>(local / NACC);
        mbar_wait(smem_u32(&tmem_empty_bar[acc]), (use & 1u) ^ 1u);  // epilogue drained this accumulator
        tc_fence_after();
        const uint32_t tacc = tmem_base + acc * Cfg::ACC_COLS;
        for (int it = 0; it < niter; ++it) {
          mbar_wait(smem_u32(&full_bar[stage]), phase);
          tc_fence_after();
          const uint32_t sa = smem_base + stage * Cfg::STAGE_BYTES;
          const uint32_t sb = sa + Cfg::A_BYTES;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint64_t bd = B_MN ? make_sdesc(sb + k * 2048, 8192, 1024) : make_sdesc(sb + k * 32, 16, 1024);
#pragma unroll
            for (int j = 0; j < MT; ++j) {
              const uint64_t ad = A_MN ? make_sdesc(sa + k * 2048, 8192, 1024)
                                       : make_sdesc(sa + j * Cfg::A_TILE + k * 32, 16, 1024);
              umma_f16(tacc + j * BN, ad, bd, idesc, (it | k) != 0 ? 1u : 0u);
            }
          }
          if (rs) {
            // A x ones^T into a 16-column side accumulator: every column = sum over K of the A row
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) {
              const uint64_t ad = A_MN ? make_sdesc(sa + k * 2048, 8192, 1024) : make_sdesc(sa + k * 32, 16, 1024);
              umma_f16(tmem_base + Cfg::RS_COL + acc * 16, ad, make_sdesc(ones_smem + k * 32, 16, 1024), idesc_rs,
                       (it | k) != 0 ? 1u : 0u);
            }
          }
          umma_commit(smem_u32(&empty_bar[stage]));  // slot reusable once these MMAs have read it
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
        umma_commit(smem_u32(&tmem_full_bar[acc]));  // accumulator complete
      }
    }
  } else {
    // ------------------------------------------------------------------------------------------ epilogue
    // 16 independent warps, no block-level barriers.  Warp (2 + ew) owns TMEM lane quarter q = warp % 4 (rows
    // 32q..32q+31 of the tile) and the 32-column chunks {ew/4, ew/4 + 4, ...}: it loads its sub-block from TMEM,
    // applies alpha / bias, transposes it through a warp-private XOR-swizzled smem tile so that 4 lanes write one
    // 64-byte row segment (full 32-byte sectors), adds the residual addend, and emits its own column-stat partial.
    const int ew = warp - 2;
    const int q = warp & 3;
    const int cc0 = ew >> 2;
    constexpr int NCHUNK = BN / 32;
    uint8_t* wstg = epi_smem + ew * Cfg::WARP_STG;                       // 2 KB tiles, 1 KB aligned (TMA SWIZZLE_64B)
    float* wbias = reinterpret_cast<float*>(epi_smem + EPI_WARPS * Cfg::WARP_STG + ew * Cfg::WARP_BIAS);
    const int sw_w = (lane >> 1) & 3;          // swizzle of the row this lane WRITES (row = lane)
    // the whole bias vector goes to shared memory once (epilogue warps only; named barrier 1)
    float* ball = reinterpret_cast<float*>(epi_smem + EPI_WARPS * (Cfg::WARP_STG + Cfg::WARP_BIAS));
    const bool bias_all = Cfg::BIAS_ALL != 0 && p.bias != nullptr && p.N <= 4096 && p.bias_stride == 0;
    if (bias_all) {
      for (int i = ew * 32 + lane; i < p.N; i += EPI_THREADS) ball[i] = p.bias[i];
      named_bar_sync(1, EPI_THREADS);
    }
    // per-CTA column-statistics accumulators: slot = n_tile * chunks_per_warp + chunk iteration (<= CS_SLOTS); the
    // statistics live on column PAIRS: lane (and lane ^ 16, a duplicate) owns columns 2*(lane&15), 2*(lane&15)+1
    constexpr int CS_SLOTS = 4;
    constexpr int CPW = (NCHUNK + 3) / 4;      // chunks per warp per tile
    float2 cs1[CS_SLOTS], cs2[CS_SLOTS];
#pragma unroll
    for (int i = 0; i < CS_SLOTS; ++i) cs1[i] = cs2[i] = make_float2(0.f, 0.f);
    const int hl = lane & 15, half = lane >> 4;
    // read side of the staging tile: this lane re-reads rows (lane>>2) + 8 i, 16-byte chunk lane&3
    const int rr0 = lane >> 2, rch = lane & 3;
    const float2 alpha2 = make_float2(p.alpha, p.alpha);
    // tile coordinates advance incrementally (tile += gridDim.x): no divisions in the loop
    int z, mn, m_tile, nt;
    fastdivmod(static_cast<int>(blockIdx.x), tiles_mn, p.mg_mn, z, mn);
    fastdivmod(mn, p.tiles_n, p.mg_n, m_tile, nt);
    int local = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++local) {
      int b = z, split = 0;
      if (p.split_k > 1) fastdivmod(z, p.split_k, p.mg_sk, b, split);
      const int n0 = nt * BN;
      const int acc = local % NACC;
      const uint32_t use = static_cast<uint32_t>(local / NACC);
      const bool use_bias = p.bias != nullptr && split == 0;
      const float* biasb = p.bias != nullptr ? p.bias + static_cast<long long>(b) * p.bias_stride : nullptr;
      // per-batch bias (not staged CTA-wide): when this warp owns a single 32-column chunk per tile, its bias slice is
      // fetched BEFORE the wait for the accumulator, so the global-load latency hides behind the tile's MMAs
      constexpr bool BIAS_EARLY = NCHUNK <= 4;
      if (BIAS_EARLY && use_bias && !bias_all && cc0 < NCHUNK) {
        const int gcb = n0 + cc0 * 32 + lane;
        wbias[lane] = gcb < p.N ? biasb[gcb] : 0.f;
      }
      mbar_wait(smem_u32(&tmem_full_bar[acc]), use & 1u);
      tc_fence_after();
#pragma unroll 1
      for (int sub = 0; sub < MT; ++sub) {       // 128-row sub-tiles of the CTA tile (one TMEM accumulator each)
      const int m0 = m_tile * BMT + sub * BM;
      const int grow = m0 + q * 32 + lane;
      const uint32_t taddr = tmem_base + acc * Cfg::ACC_COLS + sub * BN + (static_cast<uint32_t>(q * 32) << 16);
      const int rows_valid = min(32, p.M - (m0 + q * 32));   // valid rows of this warp's sub-block (may be <= 0)
      if (MT == 1 && BN <= 128 && p.rowsum != nullptr && nt == 0 && cc0 == 0) {
        // side accumulator of the row sums (one warp per 32-row quarter); read before this warp's accumulator release
        uint32_t rv[32];
        tmem_ld_32x32(tmem_base + Cfg::RS_COL + acc * 16 + (static_cast<uint32_t>(q * 32) << 16), rv);
        tmem_ld_wait();
        if (grow < p.M) {
          float* dst = p.rowsum + static_cast<long long>(b) * p.rowsum_stride + grow;
          if (p.split_k > 1) atomicAdd(dst, __uint_as_float(rv[0]));
          else *dst = __uint_as_float(rv[0]);
        }
      }
#pragma unroll 1
      for (int c = cc0; c < NCHUNK; c += 4) {
        const int gc0 = n0 + c * 32;           // first global column of this chunk
        const bool full = rows_valid >= 32 && gc0 + 32 <= p.N;
        uint32_t v[32];
        tmem_ld_32x32(taddr + c * 32, v);
        if (!BIAS_EARLY && use_bias && !bias_all) wbias[lane] = (gc0 + lane < p.N) ? biasb[gc0 + lane] : 0.f;
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (sub == MT - 1 && c + 4 >= NCHUNK && lane == 0)   // last TMEM read of this warp for the tile: release it
          mbar_arrive(smem_u32(&tmem_empty_bar[acc]));
        float2 f[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) f[j] = make_float2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
        if (p.alpha != 1.f) {
#pragma unroll
          for (int j = 0; j < 16; ++j) f[j] = mul2(f[j], alpha2);
        }
        if (use_bias) {
          // full chunks read the CTA-wide copy; a ragged last chunk (N not a multiple of 32) uses the zero-padded
          // warp-private slice
          const float* bsrc = (bias_all && gc0 + 32 <= p.N) ? ball + gc0 : wbias;
          if (bias_all && gc0 + 32 > p.N) {
            wbias[lane] = (gc0 + lane < p.N) ? ball[gc0 + lane] : 0.f;
            __syncwarp();
          }
#pragma unroll
          for (int j = 0; j < 16; j += 2) {
            const float4 bv = *reinterpret_cast<const float4*>(bsrc + 2 * j);
            f[j] = add2(f[j], make_float2(bv.x, bv.y));
            f[j + 1] = add2(f[j + 1], make_float2(bv.z, bv.w));
          }
        }
        if (p.out_kind != 0) {
          float* Df = reinterpret_cast<float*>(p.D) + static_cast<long long>(b) * p.strideD +
                      static_cast<long long>(grow) * p.ldd;
          if (grow < p.M) {
#pragma unroll
            for (int j = 0; j < 16; j += 2) {
              const int gc = gc0 + 2 * j;
              if (gc < p.N) {
                if (p.out_kind == 2) {
                  red_add_v4(Df + gc, f[j].x, f[j].y, f[j + 1].x, f[j + 1].y);
                } else {
                  *reinterpret_cast<float4*>(Df + gc) = make_float4(f[j].x, f[j].y, f[j + 1].x, f[j + 1].y);
                }
              }
            }
          }
          __syncwarp();
          continue;
        }
        // ---- bf16 output: warp-private transpose ----
        if (p.tma_store) {                       // the previous bulk store of this warp must have drained the tile
          if (lane == 0) tma_store_wait_read<0>();
          __syncwarp();
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint4 pk = make_uint4(pack_bf16(f[4 * j].x, f[4 * j].y), pack_bf16(f[4 * j + 1].x, f[4 * j + 1].y),
                                      pack_bf16(f[4 * j + 2].x, f[4 * j + 2].y),
                                      pack_bf16(f[4 * j + 3].x, f[4 * j + 3].y));
          *reinterpret_cast<uint4*>(wstg + lane * 64 + ((j ^ sw_w) << 4)) = pk;
        }
        __syncwarp();
        if (p.colstats != nullptr) {
          // sums of the stored (bf16-rounded) values over the sub-block's valid rows: each half-warp takes 16 rows,
          // each lane a column pair (16 independent 32-bit shared loads, packed fp32 accumulation), then the two
          // halves are combined; both halves end up with the pair's statistics
          float2 sa = make_float2(0.f, 0.f), sq = make_float2(0.f, 0.f);
          const uint8_t* src = wstg + half * 16 * 64 + (hl & 3) * 4;
          if (rows_valid >= 32) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float2 x = unpack_bf16(
                  *reinterpret_cast<const uint32_t*>(src + i * 64 + (((hl >> 2) ^ ((i >> 1) & 3)) << 4)));
              sa = add2(sa, x);
              sq = fma2(x, x, sq);
            }
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              if (half * 16 + i < rows_valid) {
                const float2 x = unpack_bf16(
                    *reinterpret_cast<const uint32_t*>(src + i * 64 + (((hl >> 2) ^ ((i >> 1) & 3)) << 4)));
                sa = add2(sa, x);
                sq = fma2(x, x, sq);
              }
            }
          }
          sa.x += __shfl_xor_sync(0xffffffffu, sa.x, 16);
          sa.y += __shfl_xor_sync(0xffffffffu, sa.y, 16);
          sq.x += __shfl_xor_sync(0xffffffffu, sq.x, 16);
          sq.y += __shfl_xor_sync(0xffffffffu, sq.y, 16);
          if (p.cs_accum) {
            const int slot = nt * CPW + (c >> 2);
#pragma unroll
            for (int i = 0; i < CS_SLOTS; ++i) {
              if (i == slot) {
                cs1[i] = add2(cs1[i], sa);
                cs2[i] = add2(cs2[i], sq);
              }
            }
          } else if (half == 0 && gc0 + 2 * hl < p.N) {
            float* cs = p.colstats + ((static_cast<long long>(b) * p.tiles_m + m_tile) * 4 + q) * 2 * p.N;  // MT == 1
            *reinterpret_cast<float2*>(cs + gc0 + 2 * hl) = sa;
            *reinterpret_cast<float2*>(cs + p.N + gc0 + 2 * hl) = sq;
          }
        }
        if (p.tma_store) {
          // one bulk tensor store per 32 x 32 sub-block: the staging tile is already in the SWIZZLE_64B layout the
          // tensor map expects; rows / columns beyond M / N are clipped by the TMA unit
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_3d(&tmD, smem_u32(wstg), gc0, m0 + q * 32, b);
            tma_store_commit();
          }
          continue;
        }
        bf16* Drow = reinterpret_cast<bf16*>(p.D) + static_cast<long long>(b) * p.strideD +
                     static_cast<long long>(m0 + q * 32 + rr0) * p.ldd + gc0 + rch * 8;
        const bf16* Arow = p.addend ? p.addend + static_cast<long long>(b) * p.stride_add +
                                          static_cast<long long>(m0 + q * 32 + rr0) * p.ld_add + gc0 + rch * 8
                                    : nullptr;
        const uint8_t* rsrc = wstg + rr0 * 64;
        const int gc = gc0 + rch * 8;
        uint4 adv[4];
        if (Arow != nullptr) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            adv[i] = (full || (rr0 + 8 * i < rows_valid && gc < p.N))
                         ? *reinterpret_cast<const uint4*>(Arow + static_cast<long long>(8 * i) * p.ld_add)
                         : make_uint4(0, 0, 0, 0);
          }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          // row rr0 + 8 i: (row >> 1) & 3 == (rr0 >> 1) & 3 because 8 i >> 1 is a multiple of 4
          if (full || (rr0 + 8 * i < rows_valid && gc < p.N)) {
            uint4 pk = *reinterpret_cast<const uint4*>(rsrc + i * 8 * 64 + ((rch ^ ((rr0 >> 1) & 3)) << 4));
            if (Arow != nullptr) {
              const uint32_t* a32 = reinterpret_cast<const uint32_t*>(&adv[i]);
              uint32_t* p32 = reinterpret_cast<uint32_t*>(&pk);
#pragma unroll
              for (int t = 0; t < 4; ++t) {
                const float2 s2 = add2(unpack_bf16(p32[t]), unpack_bf16(a32[t]));
                p32[t] = pack_bf16(s2.x, s2.y);
              }
            }
            *reinterpret_cast<uint4*>(Drow + static_cast<long long>(8 * i) * p.ldd) = pk;
          }
        }
        __syncwarp();                            // staging reused by the next chunk / tile
      }
      }  // sub-tiles
      if (cc0 >= NCHUNK && lane == 0)            // warps without a chunk (BN = 64) still release the accumulator
        mbar_arrive(smem_u32(&tmem_empty_bar[acc]));
      // next tile of this CTA
      nt += p.step_n;
      int carry = 0;
      if (nt >= p.tiles_n) { nt -= p.tiles_n; carry = 1; }
      m_tile += p.step_m + carry;
      carry = 0;
      if (m_tile >= p.tiles_m) { m_tile -= p.tiles_m; carry = 1; }
      z += p.step_z + carry;
    }
    if (p.tma_store && lane == 0) tma_store_wait_all<0>();
    if (p.colstats != nullptr && p.cs_accum) {
      // ONE partial row per CTA: the four warps that share a column chunk (one per 32-row quarter) combine their
      // running sums through the now idle staging tiles, in a fixed order
      __syncwarp();
      float2* xs = reinterpret_cast<float2*>(wstg);          // [slot][sum | sum of squares][16 column pairs]
      if (half == 0) {
#pragma unroll
        for (int i = 0; i < CS_SLOTS; ++i) {
          xs[(2 * i) * 16 + hl] = cs1[i];
          xs[(2 * i + 1) * 16 + hl] = cs2[i];
        }
      }
      named_bar_sync(1, EPI_THREADS);
      if ((ew & 3) == 0 && cc0 < NCHUNK && half == 0) {
        float* cs = p.colstats + static_cast<long long>(blockIdx.x) * 2 * p.N;
#pragma unroll
        for (int i = 0; i < CS_SLOTS; ++i) {
          const int nt_i = i / CPW, k = i % CPW;
          const int col = nt_i * BN + (cc0 + 4 * k) * 32 + 2 * hl;
          if (nt_i < p.tiles_n && cc0 + 4 * k < NCHUNK && col < p.N) {
            float2 t1 = make_float2(0.f, 0.f), t2 = make_float2(0.f, 0.f);
#pragma unroll
            for (int w4 = 0; w4 < 4; ++w4) {
              const float2* o = reinterpret_cast<const float2*>(wstg + w4 * Cfg::WARP_STG);
              t1 = add2(t1, o[(2 * i) * 16 + hl]);
              t2 = add2(t2, o[(2 * i + 1) * 16 + hl]);
            }
            *reinterpret_cast<float2*>(cs + col) = t1;
            *reinterpret_cast<float2*>(cs + p.N + col) = t2;
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, []() {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess) {
      fn = reinterpret_cast<EncodeTiledFn>(f);
    }
  });
  return fn;
}

// Tensor map over a bf16 operand: K-major -> dims {K, rows, batch, limb}; MN-major -> dims {rows, K, batch, limb}.
int make_operand_map(CUtensorMap* tm, const GemmOperand& op, int rows, int K, int batch, int nlimbs, int box_rows,
                     CUtensorMapDataType elem = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16) {
  EncodeTiledFn enc = get_encode_fn();
  if (enc == nullptr) return set_error(GLF_ERR_DEVICE, "cuTensorMapEncodeTiled entry point unavailable");
  if ((reinterpret_cast<uintptr_t>(op.ptr) & 15) != 0) return set_error(GLF_ERR_INVALID, "GEMM operand not 16-byte aligned");
  if (op.ld % 8 != 0) return set_error(GLF_ERR_INVALID, "GEMM leading dimension must be a multiple of 8 elements");
  if (op.batch_stride % 8 != 0 || op.limb_stride % 8 != 0)
    return set_error(GLF_ERR_INVALID, "GEMM batch/limb stride must be a multiple of 8 elements");
  const cuuint64_t inner = op.mn_major ? rows : K;
  const cuuint64_t outer = op.mn_major ? K : rows;
  const int nb = (op.batch_stride != 0) ? batch : 1;
  cuuint64_t dims[4] = {inner, outer, static_cast<cuuint64_t>(nb), static_cast<cuuint64_t>(nlimbs)};
  const cuuint64_t row_bytes = static_cast<cuuint64_t>(op.ld) * 2;
  const cuuint64_t span = outer * row_bytes;
  cuuint64_t strides[3] = {row_bytes, nb > 1 ? static_cast<cuuint64_t>(op.batch_stride) * 2 : span,
                           nlimbs > 1 ? static_cast<cuuint64_t>(op.limb_stride) * 2 : span * static_cast<cuuint64_t>(nb)};
  cuuint32_t box[4] = {64u, static_cast<cuuint32_t>(op.mn_major ? 64 : box_rows), 1u, 1u};
  cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
  CUresult r = enc(tm, elem, 4, const_cast<void*>(op.ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return set_error(GLF_ERR_INVALID, "cuTensorMapEncodeTiled failed (%d): inner=%llu outer=%llu ld=%lld", (int)r,
                     (unsigned long long)inner, (unsigned long long)outer, (long long)op.ld);
  return 0;
}

// Tensor map for bf16 OUTPUT tiles: dims {N, M, batch}, box {32 columns, 32 rows, 1}, SWIZZLE_64B — the layout of the
// epilogue's warp-private staging tile (16-byte chunk index XOR ((row >> 1) & 3)).
int make_output_map(CUtensorMap* tm, void* D, int M, int N, int batch, long long ldd, long long strideD) {
  EncodeTiledFn enc = get_encode_fn();
  if (enc == nullptr) return set_error(GLF_ERR_DEVICE, "cuTensorMapEncodeTiled entry point unavailable");
  const int nb = (strideD != 0) ? batch : 1;
  cuuint64_t dims[3] = {static_cast<cuuint64_t>(N), static_cast<cuuint64_t>(M), static_cast<cuuint64_t>(nb)};
  const cuuint64_t row_bytes = static_cast<cuuint64_t>(ldd) * 2;
  cuuint64_t strides[2] = {row_bytes, nb > 1 ? static_cast<cuuint64_t>(strideD) * 2 : row_bytes * static_cast<cuuint64_t>(M)};
  cuuint32_t box[3] = {32u, 32u, 1u};
  cuuint32_t estr[3] = {1u, 1u, 1u};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, D, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(GLF_ERR_INVALID, "cuTensorMapEncodeTiled (output) failed (%d)", (int)r);
  return 0;
}

}  // namespace

int make_operand_tmap(CUtensorMap* tm, const GemmOperand& op, int rows, int K, int batch, int nlimbs, int box_rows) {
  return make_operand_map(tm, op, rows, K, batch, nlimbs, box_rows);
}
int make_output_tmap(CUtensorMap* tm, void* D, int M, int N, int batch, long long ldd, long long strideD) {
  return make_output_map(tm, D, M, N, batch, ldd, strideD);
}

// 16-bit tensor map over [batch][outer][inner] with row pitch `ld` elements, SWIZZLE_128B, box {64, box_outer, 1, 1};
// dtype GLF_DTYPE_BF16 or GLF_DTYPE_F16
int make_tmap_bf16(CUtensorMap* tm, const void* ptr, long long inner, long long outer, long long batch, long long ld,
                   long long batch_stride, int box_outer, int dtype) {
  GemmOperand op;
  op.ptr = ptr;
  op.mn_major = 0;      // {K = inner, rows = outer}
  op.ld = ld;
  op.batch_stride = batch > 1 ? batch_stride : 0;
  return make_operand_map(tm, op, static_cast<int>(outer), static_cast<int>(inner), static_cast<int>(batch), 1, box_outer,
                          dtype == GLF_DTYPE_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
}

namespace {

template <bool A_MN, bool B_MN, int BN, int MT = 1>
int launch(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmD, GemmKParams p, int num_sms,
           int* cs_rows, cudaStream_t stream) {
  using Cfg = GemmCfg<BN, MT>;
  auto kern = gemm_kernel<A_MN, B_MN, BN, MT>;
  p.tiles_m = (p.M + BM * MT - 1) / (BM * MT);
  // per launch: the attribute is per device, and callers may drive several GPUs from one process (nn.DataParallel)
  cudaError_t attr_err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
  if (attr_err != cudaSuccess) return check_cuda(attr_err, "cudaFuncSetAttribute(gemm)");
  p.tiles_n = (p.N + BN - 1) / BN;
  const long long total = static_cast<long long>(p.tiles_m) * p.tiles_n * p.batch * p.split_k;
  if (total > 0x7fffffffLL) return set_error(GLF_ERR_INVALID, "gemm: too many tiles");
  const int grid = static_cast<int>(total < num_sms ? total : num_sms);
  // column statistics: running sums per CTA when the (n-tile, chunk) slots fit the register accumulators
  // (and the 4 * grid rows fit the documented table capacity of 4 * batch * tiles_m rows)
  auto magic = [](long long d) { return d <= 1 ? 0u : static_cast<unsigned>((1ULL << 32) / static_cast<unsigned long long>(d)); };
  p.mg_mn = magic(static_cast<long long>(p.tiles_m) * p.tiles_n);
  p.mg_n = magic(p.tiles_n);
  p.mg_sk = magic(p.split_k);
  p.cs_accum = (p.colstats != nullptr && p.tiles_n * ((BN / 32 + 3) / 4) <= 4 &&
                grid <= static_cast<long long>(p.batch) * p.tiles_m) ? 1 : 0;
  if (cs_rows != nullptr)
    *cs_rows = p.colstats == nullptr ? 0 : (p.cs_accum ? grid : p.batch * p.tiles_m * 4);
  p.step_n = grid % p.tiles_n;
  p.step_m = (grid / p.tiles_n) % p.tiles_m;
  p.step_z = grid / (p.tiles_m * p.tiles_n);
  kern<<<grid, GEMM_THREADS, Cfg::SMEM_BYTES, stream>>>(tmA, tmB, tmD, p);
  return check_cuda(cudaGetLastError(), "gemm launch");
}

template <int BN>
int launch_major(bool a_mn, bool b_mn, const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmD,
                 const GemmKParams& p, int num_sms, int* cs_rows, cudaStream_t stream) {
  if (!a_mn && !b_mn) return launch<false, false, BN>(tmA, tmB, tmD, p, num_sms, cs_rows, stream);
  if (a_mn && b_mn) return launch<true, true, BN>(tmA, tmB, tmD, p, num_sms, cs_rows, stream);
  if (a_mn) return launch<true, false, BN>(tmA, tmB, tmD, p, num_sms, cs_rows, stream);
  return launch<false, true, BN>(tmA, tmB, tmD, p, num_sms, cs_rows, stream);
}

}  // namespace

int gemm(const GemmArgs& a, cudaStream_t stream) {
  if (a.M <= 0 || a.N <= 0 || a.K <= 0 || a.batch <= 0) return set_error(GLF_ERR_INVALID, "gemm: empty problem");
  if (a.N % 8 != 0) return set_error(GLF_ERR_INVALID, "gemm: N must be a multiple of 8 (got %d)", a.N);
  if (a.out_kind < 0 || a.out_kind > 2) return set_error(GLF_ERR_INVALID, "gemm: bad out_kind");
  if (a.split_k > 1 && a.out_kind != 2) return set_error(GLF_ERR_INVALID, "gemm: split_k needs atomic output");
  if (a.out_kind != 0 && (a.addend != nullptr || a.colstats != nullptr))
    return set_error(GLF_ERR_INVALID, "gemm: addend/colstats only with bf16 output");
  if (a.ldd % 8 != 0 || (reinterpret_cast<uintptr_t>(a.D) & 15) != 0)
    return set_error(GLF_ERR_INVALID, "gemm: output must be 16-byte aligned with ldd %% 8 == 0");
  if (a.npairs < 1 || a.npairs > 6) return set_error(GLF_ERR_INVALID, "gemm: npairs out of range");
  if (a.rowsum != nullptr && a.npairs != 1) return set_error(GLF_ERR_INVALID, "gemm: rowsum needs a single operand pair");

  // Small-K products are HBM-bound: 128-wide tiles keep 2 CTAs per SM so one CTA's epilogue overlaps the other's
  // loads.  Large-K (tensor-bound, e.g. C=2048) products take the 128x256 tile.
  int BN = (a.N <= 64) ? 64 : ((a.K >= 512 && a.N % 256 == 0) ? 256 : 128);
  if (a.bn_hint == 64 || a.bn_hint == 128 || a.bn_hint == 256) BN = a.bn_hint;
  if (a.rowsum != nullptr && BN > 128) BN = 128;   // the side accumulator needs TMEM columns beyond the two stages
  int dev = 0, num_sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || num_sms <= 0)
    return set_error(GLF_ERR_DEVICE, "gemm: cannot query the SM count");
  const bool amn = a.A.mn_major != 0, bmn = a.B.mn_major != 0;
  // the big K-major products with N = 256 (U, dX of the Gram form) run on CTA pairs (glf_gemm2.cu)
  if (gemm_bres_applicable(a, num_sms)) return gemm_bres(a, num_sms, stream);
  if (gemm_pair_applicable(a, num_sms)) return gemm_pair(a, num_sms, stream);
  int nlimbsA = 1, nlimbsB = 1;
  for (int i = 0; i < a.npairs; ++i) {
    nlimbsA = a.pairA[i] + 1 > nlimbsA ? a.pairA[i] + 1 : nlimbsA;
    nlimbsB = a.pairB[i] + 1 > nlimbsB ? a.pairB[i] + 1 : nlimbsB;
  }
  CUtensorMap tmA, tmB;
  int rc = make_operand_map(&tmA, a.A, a.A.rows > 0 ? a.A.rows : a.M, a.K, a.batch, nlimbsA, BM);
  if (rc) return rc;
  rc = make_operand_map(&tmB, a.B, a.B.rows > 0 ? a.B.rows : a.N, a.K, a.batch, nlimbsB, BN);
  if (rc) return rc;

  // bf16 outputs without a residual addend leave through bulk tensor stores
  CUtensorMap tmD = tmA;
  const bool tma_store = a.out_kind == 0 && a.addend == nullptr && a.M >= 32 && a.N >= 32 && a.strideD % 8 == 0;
  if (tma_store) {
    rc = make_output_map(&tmD, a.D, a.M, a.N, a.batch, a.ldd, a.strideD);
    if (rc) return rc;
  }

  GemmKParams p;
  p.tma_store = tma_store ? 1 : 0;
  p.M = a.M; p.N = a.N; p.K = a.K; p.batch = a.batch;
  p.kb_total = (a.K + BK - 1) / BK;
  int sk = a.split_k < 1 ? 1 : a.split_k;
  if (sk > p.kb_total) sk = p.kb_total;
  p.kb_per_split = (p.kb_total + sk - 1) / sk;
  p.split_k = (p.kb_total + p.kb_per_split - 1) / p.kb_per_split;
  p.npairs = a.npairs;
  for (int i = 0; i < 6; ++i) { p.pairA[i] = a.pairA[i]; p.pairB[i] = a.pairB[i]; }
  p.a_batched = a.A.batch_stride != 0;
  p.b_batched = a.B.batch_stride != 0;
  p.alpha = a.alpha;
  p.bias = a.bias;
  p.out_kind = a.out_kind;
  p.D = a.D; p.ldd = a.ldd; p.strideD = a.strideD;
  p.addend = a.addend; p.ld_add = a.ld_add; p.stride_add = a.stride_add;
  p.colstats = a.colstats;
  p.bias_stride = a.bias != nullptr ? a.bias_stride : 0;
  p.rowsum = a.rowsum;
  p.rowsum_stride = a.rowsum_stride;
  p.cs_accum = 0;
  p.tiles_m = gemm_tiles_m(a.M);
  p.tiles_n = 0;  // set per tile shape in launch()
  // 256-row super-tiles (MT = 2) for the big K-major products: halves the B-operand traffic per output row.  The
  // column statistics need the per-CTA running-sum mode there (one partial row per CTA).
  bool mt2 = !amn && BN == 128 && a.rowsum == nullptr && a.M >= 1024;
  if (mt2 && a.colstats != nullptr) {
    const long long tm2 = (a.M + 2 * BM - 1) / (2 * BM), tn = (a.N + BN - 1) / BN;
    const long long total = tm2 * tn * a.batch * p.split_k;
    const long long grid = total < num_sms ? total : num_sms;
    mt2 = tn * ((BN / 32 + 3) / 4) <= 4 && grid <= static_cast<long long>(a.batch) * tm2;
  }
  if (mt2)
    return bmn ? launch<false, true, 128, 2>(tmA, tmB, tmD, p, num_sms, a.colstats_rows, stream)
               : launch<false, false, 128, 2>(tmA, tmB, tmD, p, num_sms, a.colstats_rows, stream);
  switch (BN) {
    case 64: return launch_major<64>(amn, bmn, tmA, tmB, tmD, p, num_sms, a.colstats_rows, stream);
    case 128: return launch_major<128>(amn, bmn, tmA, tmB, tmD, p, num_sms, a.colstats_rows, stream);
    default: return launch_major<256>(amn, bmn, tmA, tmB, tmD, p, num_sms, a.colstats_rows, stream);
  }
}

}  // namespace glf
