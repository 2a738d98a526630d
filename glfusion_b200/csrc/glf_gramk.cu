// glf_gramk.cu — token contraction of the Gram form: per sequence b,  D_b = A_b^T X_b  ([C x C], C = 128 or 256) with
// A = X (S = X^T X, forward) or A = dV (R = dV^T X, backward), plus the column sums of A.
//
// The generic tile GEMM (glf_gemm.cu) computes this product as four 128 x 128 tiles per sequence, so every 64-token
// block of A and X is pulled from L2 twice and the kernel ends up bound by the L2 -> SM fabric (ncu: tensor pipe 43 %,
// DRAM 31 %, profiles/r01_gram_gemm_ncu_brief.txt).  Here ONE CTA owns a whole sequence (or a K split of it): each
// 64-token block [64 x C] of A and of X is loaded exactly once (TMA, SWIZZLE_128B, MN-major), the C x C fp32 result
// lives in TMEM (C = 256: two 128-lane accumulators x 256 columns = all 512 columns), and the operands are read
// straight from HBM once: the S product is tensor-bound, the R product HBM-bound (two inputs).
//
//   warp 0      TMA producer: per k-block C/64 boxes of A (+ C/64 boxes of X unless A == X) into a 3-stage ring
//   warp 1      MMA issuer: tcgen05.mma M=128, N=C, K=16, both operands MN-major, C/128 accumulators
//   warps 2..9  during the main loop: column sums of A read from the staged blocks (thread = channel); afterwards the
//               epilogue: tcgen05.ld -> bf16 rows of the augmented [Ca x Ca] matrix, or fp32 red.add for split-K
#include <cstdio>
#include <cstdlib>

#include "glf_internal.h"
#include "glf_ptx.cuh"

namespace glf {

namespace {

constexpr int GK_THREADS = 64 + 256;
constexpr int GK_STAGES = 3;                       // A != X: three stages of (A block + X block)
constexpr int GK_MAX_STAGES = 6;                   // A == X: the same ring holds six single-block stages
constexpr uint32_t GK_BLK = 64 * 256 * 2;          // one operand block: 64 tokens x 256 channels (4 boxes of 64 x 64)
constexpr uint32_t GK_STAGE = 2 * GK_BLK;          // A block + X block
constexpr uint32_t GK_SMEM = GK_STAGES * GK_STAGE + 1024;

// Debug aid (GLF_GRAM_TRACE=1): SM clock of CTA 0 at a few points, printed by the host after the launch.
__device__ long long g_gram_trace[8];
#define GK_TRACE(i)                                             \
  do {                                                          \
    if (p.trace && blockIdx.x == 0) g_gram_trace[i] = clock64(); \
  } while (0)

struct GramKParams {
  int B, N, C, Ca;
  int ksplit, kb_total, kb_per_split;
  int same;        // A == X: the X block is not loaded, the B operand is the A block
  int sym;         // same && C == 256 && ksplit == 1: the lower-left 128 x 128 block is mirrored, not computed
  bf16* out;       // ksplit == 1: [B][Ca][Ca] bf16, rows/cols < C written
  float* outf;     // ksplit  > 1: [B][C][C] fp32, atomically accumulated (zeroed by the caller)
  float* rowsum;   // [B][C] column sums of A (stored, or atomically accumulated when ksplit > 1)
  int slabs;       // ksplit > 1: split s stores into slab s (outf + s [B][C][C], rowsum + s [B][C]) instead of atomics
  const float* rowscale;   // optional [C]: bf16 output row r is scaled by rowscale[r] (ksplit == 1 path)
  // ksplit == 1: the homogeneous border of the augmented matrix is written here as well (no separate launch):
  //   column C = rowscale * column sums of A, row C = rowv (or the column sums when rowv is null), corner, zero padding
  const float* rowv;       // optional [B][C]
  float corner;
  int border;              // 1: write the border (needs Ca >= C + 1)
  // CTAs >= nwork are not contraction work: they convert the fp32 weight masters to the bf16 operands of the chain
  // that follows (W~{theta,phi,g} = [W | b | 0] as [3][Ci][Ca], Wz as [C][Ci]) — the launch the forward used to spend on it
  int nwork, nprep;
  GramPrep prep;
  int trace;
};

__global__ void __launch_bounds__(GK_THREADS, 1)
    gram_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmX, const GramKParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t full_bar[GK_MAX_STAGES];
  __shared__ uint64_t empty_bar[GK_MAX_STAGES];
  __shared__ uint64_t tmem_full_bar;
  __shared__ uint32_t tmem_holder;

  if (static_cast<int>(blockIdx.x) >= p.nwork) {            // weight preparation rides along (whole CTA, no barriers used)
    const GramPrep& q = p.prep;
    const int naug = 3 * q.Ci * q.Ca, nz = q.C * q.Ci;
    for (int i = (blockIdx.x - p.nwork) * GK_THREADS + threadIdx.x; i < naug + nz; i += p.nprep * GK_THREADS) {
      if (i < naug) {
        const int m = i / (q.Ci * q.Ca), r = (i / q.Ca) % q.Ci, c = i % q.Ca;
        const float* W = m == 0 ? q.tw : (m == 1 ? q.pw : q.gw);
        const float* bb = m == 0 ? q.tb : (m == 1 ? q.pb : q.gb);
        const float v = c < q.C ? W[static_cast<size_t>(r) * q.C + c] : (c == q.C ? bb[r] : 0.f);
        q.waug[i] = __float2bfloat16(v);
      } else {
        q.wzb[i - naug] = __float2bfloat16(q.wz[i - naug]);
      }
    }
    return;
  }
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x / p.ksplit;
  const int split = blockIdx.x - b * p.ksplit;
  const int kb0 = split * p.kb_per_split;
  const int nkb = min(p.kb_total, kb0 + p.kb_per_split) - kb0;
  const int nbox = p.C / 64;     // 64-channel boxes per block
  const int MT = p.C / 128;      // 128-row accumulators
  // S = X^T X loads one block per k-step: twice the stages in the same ring (more bytes in flight per SM: the product
  // is bound by the latency of its own HBM stream otherwise)
  const int nstages = p.same ? GK_MAX_STAGES : GK_STAGES;
  const uint32_t stage_bytes = p.same ? GK_BLK : GK_STAGE;

  if (threadIdx.x == 0) {
    GK_TRACE(0);
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmX);
#pragma unroll
    for (int s = 0; s < GK_MAX_STAGES; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      // MMA commit + the eight column-sum warps (symmetric S: the column sums come from the tensor core as well)
      mbar_init(smem_u32(&empty_bar[s]), p.sym ? 1 : 1 + 8);
    }
    mbar_init(smem_u32(&tmem_full_bar), 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_holder), 512);
  __shared__ __align__(1024) uint8_t ones_tile[2048];          // K-major [16 rows][64 k] of bf16 1.0 (swizzle-invariant)
  if (p.sym) {
    for (int i = threadIdx.x; i < 512; i += GK_THREADS) reinterpret_cast<uint32_t*>(ones_tile)[i] = 0x3F803F80u;
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_holder;

  if (warp == 0) {
    if (elect_one()) {
      const uint32_t bytes = static_cast<uint32_t>(nbox) * 8192u * (p.same ? 1u : 2u);
      int stage = 0;
      uint32_t phase = 0;
      for (int it = 0; it < nkb; ++it) {
        const int k0 = (kb0 + it) * 64;
        const uint32_t fb = smem_u32(&full_bar[stage]);
        mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1u);
        mbar_expect_tx(fb, bytes);
        const uint32_t sa = smem_base + stage * stage_bytes;
        for (int j = 0; j < nbox; ++j) tma_load_4d(&tmA, fb, sa + j * 8192, j * 64, k0, b, 0);
        if (!p.same)
          for (int j = 0; j < nbox; ++j) tma_load_4d(&tmX, fb, sa + GK_BLK + j * 8192, j * 64, k0, b, 0);
        if (++stage == nstages) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      const uint32_t idesc = make_idesc_bf16(128, p.C, true, true);
      const uint32_t idesc_half = make_idesc_bf16(128, 128, true, true);
      const uint32_t idesc_ones = make_idesc_bf16(128, 16, true, false);
      int stage = 0;
      uint32_t phase = 0;
      GK_TRACE(1);
      for (int it = 0; it < nkb; ++it) {
        mbar_wait(smem_u32(&full_bar[stage]), phase);
        if (it == 0) GK_TRACE(2);
        if (it == nkb / 2) GK_TRACE(3);
        tc_fence_after();
        const uint32_t sa = smem_base + stage * stage_bytes;
        const uint32_t sb = p.same ? sa : sa + GK_BLK;
        if (p.sym) {
          // S = X^T X is symmetric: rows 0..127 take all 256 columns, rows 128..255 only columns 128..255; the
          // epilogue mirrors the upper-right block into the lower-left one (a quarter of the MMA work and of its
          // shared-memory operand traffic saved: the kernel is bound by shared-memory bandwidth, not by the tensor pipe)
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            umma_f16(tmem_base, make_sdesc(sa + k * 2048, 8192, 1024), make_sdesc(sa + k * 2048, 8192, 1024), idesc,
                     (it | k) != 0 ? 1u : 0u);
            umma_f16(tmem_base + 256 + 128, make_sdesc(sa + 16384 + k * 2048, 8192, 1024),
                     make_sdesc(sa + 16384 + k * 2048, 8192, 1024), idesc_half, (it | k) != 0 ? 1u : 0u);
            // column sums of X = X^T 1: both 128-channel halves against the ones tile, into the TMEM columns the
            // mirrored block leaves free (256 .. 271 and 272 .. 287)
            const uint64_t od = make_sdesc(smem_u32(ones_tile) + k * 32, 16, 1024);
            umma_f16(tmem_base + 256, make_sdesc(sa + k * 2048, 8192, 1024), od, idesc_ones, (it | k) != 0 ? 1u : 0u);
            umma_f16(tmem_base + 256 + 16, make_sdesc(sa + 16384 + k * 2048, 8192, 1024), od, idesc_ones,
                     (it | k) != 0 ? 1u : 0u);
          }
        } else {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint64_t bd = make_sdesc(sb + k * 2048, 8192, 1024);
            for (int mt = 0; mt < MT; ++mt) {
              const uint64_t ad = make_sdesc(sa + mt * 16384 + k * 2048, 8192, 1024);
              umma_f16(tmem_base + mt * p.C, ad, bd, idesc, (it | k) != 0 ? 1u : 0u);
            }
          }
        }
        umma_commit(smem_u32(&empty_bar[stage]));
        if (++stage == nstages) { stage = 0; phase ^= 1u; }
      }
      umma_commit(smem_u32(&tmem_full_bar));
      GK_TRACE(4);
    }
  } else {
    // ---- column sums of A from the staged blocks: thread = (channel pair cp, half of the 64 rows); 32-bit loads (the
    //      kernel is bound by shared-memory bandwidth: 2-byte loads waste half of every wavefront)
    const int t = threadIdx.x - 64;
    __shared__ float cs_x[2][256];
    // column sum `cs` of channel `ch`: stored (or atomically added for a token split), plus the homogeneous border
    auto emit_colsum = [&](int ch, float cs) {
      float* dst = p.rowsum + static_cast<long long>(b) * p.C + ch;
      if (p.ksplit > 1) {
        if (p.slabs) dst[static_cast<long long>(split) * p.B * p.C] = cs;
        else atomicAdd(dst, cs);
        return;
      }
      *dst = cs;
      if (!p.border) return;
      // border of the augmented matrix: out[ch][C .. Ca) = {scaled column sum, 0 ...}; out[C][ch] = rowv or the sum
      bf16* M = p.out + static_cast<long long>(b) * p.Ca * p.Ca;
      const float rs = p.rowscale != nullptr ? p.rowscale[ch] : 1.f;
      if (p.Ca - p.C == 8) {
        *reinterpret_cast<uint4*>(M + static_cast<long long>(ch) * p.Ca + p.C) = make_uint4(pack_bf16(cs * rs, 0.f), 0u, 0u, 0u);
      } else {
        for (int j = p.C; j < p.Ca; ++j) M[static_cast<long long>(ch) * p.Ca + j] = __float2bfloat16(j == p.C ? cs * rs : 0.f);
      }
      M[static_cast<long long>(p.C) * p.Ca + ch] =
          __float2bfloat16(p.rowv != nullptr ? p.rowv[static_cast<long long>(b) * p.C + ch] : cs);
      if (ch == 0)
        for (int j = p.C; j < p.Ca; ++j)
          M[static_cast<long long>(p.C) * p.Ca + j] = __float2bfloat16(j == p.C ? p.corner : 0.f);
    };
    if (!p.sym) {
      const int cp = t & 127, rh = t >> 7;                       // channels 2 cp, 2 cp + 1 ; rows 32 rh .. 32 rh + 31
      const int ch = 2 * cp;
      const uint32_t off0 = static_cast<uint32_t>(ch >> 6) * 8192u + static_cast<uint32_t>(ch & 7) * 2u;
      const uint32_t chunk = static_cast<uint32_t>((ch & 63) >> 3);
      float2 a2 = make_float2(0.f, 0.f), b2 = make_float2(0.f, 0.f);
      int stage = 0;
      uint32_t phase = 0;
      for (int it = 0; it < nkb; ++it) {
        mbar_wait(smem_u32(&full_bar[stage]), phase);
        if (ch < p.C) {
          const uint8_t* blk = smem_gen + stage * stage_bytes + off0 + rh * 32 * 128;
#pragma unroll 8
          for (int k = 0; k < 32; k += 2) {
            a2 = add2(a2, unpack_bf16(*reinterpret_cast<const uint32_t*>(blk + k * 128 + ((chunk ^ (k & 7)) << 4))));
            b2 = add2(b2, unpack_bf16(*reinterpret_cast<const uint32_t*>(blk + (k + 1) * 128 + ((chunk ^ ((k + 1) & 7)) << 4))));
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&empty_bar[stage]));
        if (++stage == nstages) { stage = 0; phase ^= 1u; }
      }
      const float2 tot = add2(a2, b2);
      if (ch < p.C) {
        cs_x[rh][ch] = tot.x;
        cs_x[rh][ch + 1] = tot.y;
      }
      named_bar_sync(1, 256);
      const float acc0 = t < p.C ? cs_x[0][t] : 0.f, acc1 = t < p.C ? cs_x[1][t] : 0.f;
      if (t < p.C) emit_colsum(t, acc0 + acc1);
    }
    // ---- epilogue: warp (mt, q) owns TMEM lanes 32q..32q+31 of accumulator mt = output rows 128 mt + 32 q + lane
    const int q = warp & 3;
    const int mt = (warp - 2) >> 2;
    mbar_wait(smem_u32(&tmem_full_bar), 0);
    if (threadIdx.x == 64) GK_TRACE(5);
    tc_fence_after();
    if (mt < MT) {
      const int row = mt * 128 + q * 32 + lane;
      const float rsc = (p.rowscale != nullptr && p.ksplit == 1) ? p.rowscale[row] : 1.f;
      if (p.sym) {            // the column sums sit in TMEM columns 256 + 16 mt (every column of the group holds them)
        uint32_t sv[32];
        tmem_ld_32x32(tmem_base + 256 + (static_cast<uint32_t>(q * 32) << 16), sv);
        tmem_ld_wait();
        emit_colsum(row, __uint_as_float(sv[mt * 16]));
      }
      const uint32_t taddr = tmem_base + mt * p.C + (static_cast<uint32_t>(q * 32) << 16);
      // ksplit == 1: the bf16 rows are staged in the (now idle) ring, row pitch 528 bytes (= Ca of C = 256: successive
      // rows are four banks apart), and leave with coalesced 16-byte stores below: a row per thread straight from
      // registers touched 32 lines per store instruction.  Symmetric S: rows 128..255 hold only columns 128..255 in
      // TMEM; rows 0..127 also write their columns 128..255 TRANSPOSED into the staged rows 128..255 (the mirror).
      constexpr uint32_t STG_PITCH = 528;
      uint8_t* stg = const_cast<uint8_t*>(smem_gen);
      for (int c = (p.sym && mt == 1) ? 4 : 0; c < p.C / 32; ++c) {
        uint32_t v[32];
        tmem_ld_32x32(taddr + c * 32, v);
        tmem_ld_wait();
        if (p.ksplit > 1) {
          float* dst = p.outf + (static_cast<long long>(b) * p.C + row) * p.C + c * 32;
          if (p.slabs) {
            dst += static_cast<long long>(split) * p.B * p.C * p.C;
#pragma unroll
            for (int j = 0; j < 32; j += 4)
              *reinterpret_cast<float4*>(dst + j) = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]),
                                                                __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
          } else {
#pragma unroll
            for (int j = 0; j < 32; j += 4)
              asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + j), "f"(__uint_as_float(v[j])),
                           "f"(__uint_as_float(v[j + 1])), "f"(__uint_as_float(v[j + 2])), "f"(__uint_as_float(v[j + 3]))
                           : "memory");
          }
        } else {
          uint8_t* dst = stg + static_cast<uint32_t>(row) * STG_PITCH + c * 64;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint4 pk = make_uint4(pack_bf16(rsc * __uint_as_float(v[8 * j]), rsc * __uint_as_float(v[8 * j + 1])),
                                        pack_bf16(rsc * __uint_as_float(v[8 * j + 2]), rsc * __uint_as_float(v[8 * j + 3])),
                                        pack_bf16(rsc * __uint_as_float(v[8 * j + 4]), rsc * __uint_as_float(v[8 * j + 5])),
                                        pack_bf16(rsc * __uint_as_float(v[8 * j + 6]), rsc * __uint_as_float(v[8 * j + 7])));
            *reinterpret_cast<uint4*>(dst + 16 * j) = pk;
          }
          if (p.sym && mt == 0 && c >= 4) {
            uint8_t* tdst = stg + row * 2;          // element (col, row) of the staged matrix, col = 32 c + j >= 128
#pragma unroll
            for (int j = 0; j < 32; ++j)
              *reinterpret_cast<bf16*>(tdst + static_cast<uint32_t>(c * 32 + j) * STG_PITCH) =
                  __float2bfloat16(__uint_as_float(v[j]));
          }
        }
      }
    }
    if (p.ksplit == 1 && p.C == 256) {
      named_bar_sync(1, 256);
      // 256 rows x 512 bytes -> global rows of pitch Ca; a warp moves one row per iteration
      uint8_t* gout = reinterpret_cast<uint8_t*>(p.out + static_cast<long long>(b) * p.Ca * p.Ca);
      const uint8_t* stg = smem_gen;
#pragma unroll 4
      for (int it = 0; it < 32; ++it) {
        const int r = it * 8 + (warp - 2);
        *reinterpret_cast<uint4*>(gout + static_cast<long long>(r) * p.Ca * 2 + lane * 16) =
            *reinterpret_cast<const uint4*>(stg + static_cast<uint32_t>(r) * 528u + lane * 16);
      }
    } else if (p.ksplit == 1) {
      named_bar_sync(1, 256);
      // C = 128: 128 rows x 256 bytes
      uint8_t* gout = reinterpret_cast<uint8_t*>(p.out + static_cast<long long>(b) * p.Ca * p.Ca);
      const uint8_t* stg = smem_gen;
      for (int idx = t; idx < 128 * 16; idx += 256) {
        const int r = idx >> 4, ch = idx & 15;
        *reinterpret_cast<uint4*>(gout + static_cast<long long>(r) * p.Ca * 2 + ch * 16) =
            *reinterpret_cast<const uint4*>(stg + static_cast<uint32_t>(r) * 528u + ch * 16);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) GK_TRACE(6);
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

}  // namespace

bool gram_contraction_supported(int C) { return C == 128 || C == 256; }

// ksplit == 1: out_aug rows / columns < C (bf16, ld = Ca, row r scaled by rowscale[r] if given) and, with `border`, the
// homogeneous border (column C = scaled column sums of A, row C = rowv or the column sums, corner, zero padding);
// ksplit > 1: fp32 accumulation into `scratch` (zeroed here, unscaled) for gram_assemble_aug.
// rowsum = column sums of A (unscaled).
int gram_contraction(const bf16* A, const bf16* X, bf16* out_aug, float* scratch, float* rowsum, const float* rowscale,
                     const float* rowv, float corner, int border, int B, int N, int C, int Ca, int ksplit,
                     cudaStream_t stream, const GramPrep* prep, const SplitSlab* slab) {
  if (!gram_contraction_supported(C)) return set_error(GLF_ERR_UNSUPPORTED, "gram_contraction: C must be 128 or 256");
  CUtensorMap tmA, tmX;
  int rc = make_tmap_bf16(&tmA, A, C, N, B, C, static_cast<long long>(N) * C, 64);
  if (rc) return rc;
  rc = make_tmap_bf16(&tmX, X, C, N, B, C, static_cast<long long>(N) * C, 64);
  if (rc) return rc;
  GramKParams p;
  p.B = B; p.N = N; p.C = C; p.Ca = Ca;
  p.kb_total = (N + 63) / 64;
  int ks = ksplit < 1 ? 1 : ksplit;
  if (ks > p.kb_total) ks = p.kb_total;
  p.kb_per_split = (p.kb_total + ks - 1) / ks;
  p.ksplit = (p.kb_total + p.kb_per_split - 1) / p.kb_per_split;
  p.same = (A == X) ? 1 : 0;
  p.sym = (p.same && C == 256 && p.ksplit == 1 && rowscale == nullptr && out_aug != nullptr) ? 1 : 0;
  p.out = out_aug; p.outf = scratch; p.rowsum = rowsum; p.rowscale = rowscale;
  p.rowv = rowv; p.corner = corner;
  p.border = (border && Ca > C) ? 1 : 0;
  p.slabs = (slab != nullptr && slab->on && p.ksplit > 1) ? 1 : 0;
  const long long BCC = static_cast<long long>(B) * C * C;
  if (p.slabs) {
    if (slab->p == nullptr || slab->floats < gram_slab_floats(B, N, C, ksplit))
      return set_error(GLF_ERR_WORKSPACE, "gram_contraction: deterministic slab scratch too small");
    p.outf = slab->p;
    p.rowsum = slab->p + p.ksplit * BCC;
  } else if (p.ksplit > 1) {
    rc = check_cuda(cudaMemsetAsync(scratch, 0, sizeof(float) * B * C * C, stream), "memset S");
    if (rc) return rc;
    rc = check_cuda(cudaMemsetAsync(rowsum, 0, sizeof(float) * B * C, stream), "memset s");
    if (rc) return rc;
  }
  cudaError_t e = cudaFuncSetAttribute(gram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GK_SMEM);
  if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(gram)");
  const long long grid = static_cast<long long>(B) * p.ksplit;
  if (grid > 0x7fffffffLL) return set_error(GLF_ERR_INVALID, "gram_contraction: too many work items");
  p.nwork = static_cast<int>(grid);
  p.nprep = 0;
  p.prep = GramPrep{};
  if (prep != nullptr) {
    p.prep = *prep;
    p.nprep = 20;          // ~134 K elements at C = 256: 21 per thread
  }
  {
    const char* et = getenv("GLF_GRAM_TRACE");
    p.trace = (et && et[0] == '1') ? 1 : 0;
  }
  gram_kernel<<<static_cast<int>(grid) + p.nprep, GK_THREADS, GK_SMEM, stream>>>(tmA, tmX, p);
  rc = check_cuda(cudaGetLastError(), "gram_contraction launch");
  if (rc == 0 && p.slabs) {   // the split slabs summed in split order: S into scratch, the column sums into rowsum
    rc = slab_reduce(p.outf, p.ksplit, BCC, scratch, B * C, C, C, 0, 1, 0, stream);
    if (rc == 0) rc = slab_reduce(p.rowsum, p.ksplit, static_cast<long long>(B) * C, rowsum, B, C, C, 0, 1, 0, stream);
  }
  if (rc == 0 && p.trace) {      // debug only: synchronises the stream
    long long t[8] = {0};
    cudaStreamSynchronize(stream);
    cudaMemcpyFromSymbol(t, g_gram_trace, sizeof(t));
    fprintf(stderr, "[gram trace same=%d sym=%d] first block landed +%lld, half of the k-blocks +%lld, last MMA issued +%lld, "
                    "accumulator complete +%lld, CTA done +%lld cycles (k loop entered +%lld)\n",
            p.same, p.sym, t[2] - t[0], t[3] - t[0], t[4] - t[0], t[5] - t[0], t[6] - t[0], t[1] - t[0]);
  }
  return rc;
}

}  // namespace glf
