// glf_gate.cu — the MLFM-specific work of the reference call site (R/models/ours.py:1802-1820, 1826-1827):
// centre-aware gate a = sigmoid(w * max_c sigmoid(cls) * sigmoid(ctr)), f4_local = f4 * a, and the view concat
// cat([f4_v.unsqueeze(2)], dim=2) for both the global (ungated) and local (gated) inputs.  In the reference this is
// ~10 element-wise / copy kernels per view; here one HBM-bound pass reads each per-view NCHW feature map once,
// transposes it through shared memory and writes both token-major [B, V*h*w, C] operands with 128-bit stores.
// The backward is the mirror pass: df4 = dXg + a * dXl (back to NCHW) plus the gate gradient da = sum_c f4 * dXl
// chained through the two sigmoids / the class max to the logits.
// f4 / df4 may be bf16, fp16 or fp32; the token-major operands are bf16 (fp32 for the F32X3 arm).  fp16 f4 is converted
// where it is read and df4 rounded to fp16 where it is written: the fp16 forms move the same bytes as the bf16 ones.
#include <type_traits>

#include "glf_internal.h"
#include "glf_ptx.cuh"

namespace glf {

namespace {

constexpr int MAXV = 8;
struct ViewPtrs {
  const void* f4[MAXV];
  const float* cls[MAXV];
  const float* ctr[MAXV];
  void* df4[MAXV];
  float* dcls[MAXV];
  float* dctr[MAXV];
};

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + __expf(-x)); }

template <typename T>
__device__ __forceinline__ float ldf(const T* p) { return static_cast<float>(*p); }
// two adjacent spatial positions of one channel (NCHW side), 4-byte / 8-byte accesses
__device__ __forceinline__ void ld2(const bf16* p, float& a, float& b) {
  const float2 t = unpack_bf16(*reinterpret_cast<const uint32_t*>(p));
  a = t.x; b = t.y;
}
__device__ __forceinline__ void ld2(const f16* p, float& a, float& b) {
  const float2 t = unpack2<f16>(*reinterpret_cast<const uint32_t*>(p));
  a = t.x; b = t.y;
}
__device__ __forceinline__ void ld2(const float* p, float& a, float& b) {
  const float2 t = *reinterpret_cast<const float2*>(p);
  a = t.x; b = t.y;
}
__device__ __forceinline__ void st2(bf16* p, float a, float b) { *reinterpret_cast<uint32_t*>(p) = pack_bf16(a, b); }
__device__ __forceinline__ void st2(f16* p, float a, float b) { *reinterpret_cast<uint32_t*>(p) = pack2<f16>(a, b); }
__device__ __forceinline__ void st2(float* p, float a, float b) { *reinterpret_cast<float2*>(p) = make_float2(a, b); }
// eight consecutive channels of one token (token-major side)
__device__ __forceinline__ void st8(bf16* p, const float (&f)[8]) {
  *reinterpret_cast<uint4*>(p) =
      make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
}
__device__ __forceinline__ void st8(f16* p, const float (&f)[8]) {
  *reinterpret_cast<uint4*>(p) =
      make_uint4(pack2<f16>(f[0], f[1]), pack2<f16>(f[2], f[3]), pack2<f16>(f[4], f[5]), pack2<f16>(f[6], f[7]));
}
__device__ __forceinline__ void st8(float* p, const float (&f)[8]) {
  *reinterpret_cast<float4*>(p) = make_float4(f[0], f[1], f[2], f[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(f[4], f[5], f[6], f[7]);
}
__device__ __forceinline__ void ld8(const bf16* p, float (&f)[8]) {
  const uint4 v = *reinterpret_cast<const uint4*>(p);
  const uint32_t* u = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = unpack_bf16(u[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ void ld8(const float* p, float (&f)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p);
  const float4 b = *reinterpret_cast<const float4*>(p + 4);
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w;
  f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}

// grid: (ceil(hw/64), C/64 rounded up, B*V) ; block 256
template <typename TIO, int VEC, typename TX>
__global__ void __launch_bounds__(256)
    gate_concat_fwd_kernel(const ViewPtrs vp, TX* __restrict__ xg, TX* __restrict__ xl, float* __restrict__ gate,
                           int C, int V, int hw, int ncls, float weight) {
  __shared__ float tile[64][65];
  __shared__ float a_sm[64];
  const int bv = blockIdx.z, b = bv / V, v = bv % V;
  const int p0 = blockIdx.x * 64, c0 = blockIdx.y * 64;
  const TIO* f4 = reinterpret_cast<const TIO*>(vp.f4[v]) + static_cast<long long>(b) * C * hw;
  if (threadIdx.x < 64) {
    const int p = p0 + threadIdx.x;
    float a = 0.f;
    if (p < hw) {
      const float* cl = vp.cls[v] + static_cast<long long>(b) * ncls * hw + p;
      float lmax = cl[0];
      for (int k = 1; k < ncls; ++k) lmax = fmaxf(lmax, cl[static_cast<long long>(k) * hw]);
      const float m = sigmoidf_(lmax);  // max_c sigmoid(l_c) == sigmoid(max_c l_c)
      const float c = sigmoidf_(vp.ctr[v][static_cast<long long>(b) * hw + p]);
      a = sigmoidf_(weight * m * c);
      if (blockIdx.y == 0) gate[static_cast<long long>(bv) * hw + p] = a;
    }
    a_sm[threadIdx.x] = a;
  }
  if (VEC == 2) {  // hw even: every (c, even p) address is 4-byte aligned
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
    for (int i = ty; i < 64; i += 8) {
      const int c = c0 + i, p = p0 + 2 * tx;
      float a = 0.f, b = 0.f;
      if (c < C && p < hw) ld2(f4 + static_cast<long long>(c) * hw + p, a, b);
      tile[i][2 * tx] = a;
      tile[i][2 * tx + 1] = b;
    }
  } else {
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
    for (int i = ty; i < 64; i += 4) {
      const int c = c0 + i, p = p0 + tx;
      tile[i][tx] = (c < C && p < hw) ? ldf(f4 + static_cast<long long>(c) * hw + p) : 0.f;
    }
  }
  __syncthreads();
  // write: 8 lanes x 16 B cover the 64 channels of one token row
  const int chunk = threadIdx.x & 7, pr = threadIdx.x >> 3;  // 32 rows per pass
  for (int pp = pr; pp < 64; pp += 32) {
    const int p = p0 + pp, c = c0 + chunk * 8;
    if (p < hw && c < C) {
      float f[8], g[8];
      const float a = a_sm[pp];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        f[i] = tile[chunk * 8 + i][pp];
        g[i] = f[i] * a;
      }
      const long long o = (static_cast<long long>(b) * V * hw + static_cast<long long>(v) * hw + p) * C + c;
      st8(xg + o, f);
      st8(xl + o, g);
    }
  }
}

// grid: (ceil(hw/64), ceil(C/64), B*V) ; block 256.  Each block handles one 64-position x 64-channel tile:
// df4 = dXg + a * dXl back to NCHW, and its partial of the gate gradient da[p] = sum_c f4[c,p] * dXl[p,c], written to
// da_part[c_tile][b,v,p] (reduced in fixed order by gate_finish_kernel: deterministic, no atomics).
template <typename TIO, int VEC, typename TX>
__global__ void __launch_bounds__(256)
    gate_concat_bwd_kernel(const ViewPtrs vp, const float* __restrict__ gate, const TX* __restrict__ dxg,
                           const TX* __restrict__ dxl, float* __restrict__ da_part, int C, int V, int hw) {
  __shared__ float tg[64][65];
  __shared__ float tl[64][65];
  __shared__ float a_sm[64];
  __shared__ float da_sm[8][64];
  const int bv = blockIdx.z, b = bv / V, v = bv % V;
  const int p0 = blockIdx.x * 64, c0 = blockIdx.y * 64;
  const TIO* f4 = reinterpret_cast<const TIO*>(vp.f4[v]) + static_cast<long long>(b) * C * hw;
  TIO* df4 = reinterpret_cast<TIO*>(vp.df4[v]) + static_cast<long long>(b) * C * hw;
  if (threadIdx.x < 64) {
    const int p = p0 + threadIdx.x;
    a_sm[threadIdx.x] = p < hw ? gate[static_cast<long long>(bv) * hw + p] : 0.f;
  }
  // NCHW side mapping: VEC==2 -> 32 position pairs x 8 channel rows ; VEC==1 -> 64 positions x 4 channel rows
  const int tx = VEC == 2 ? (threadIdx.x & 31) : (threadIdx.x & 63);
  const int ty = VEC == 2 ? (threadIdx.x >> 5) : (threadIdx.x >> 6);
  constexpr int NY = VEC == 2 ? 8 : 4;
  // issue the NCHW-side f4 loads first: they do not depend on shared memory
  float fv0[64 / NY], fv1[64 / NY];
#pragma unroll
  for (int k = 0; k < 64 / NY; ++k) {
    const int i = ty + k * NY;
    const int c = c0 + i;
    fv0[k] = fv1[k] = 0.f;
    if (VEC == 2) {
      const int p = p0 + 2 * tx;
      if (c < C && p < hw) ld2(f4 + static_cast<long long>(c) * hw + p, fv0[k], fv1[k]);
    } else {
      const int p = p0 + tx;
      if (c < C && p < hw) fv0[k] = ldf(f4 + static_cast<long long>(c) * hw + p);
    }
  }
  {
    const int chunk = threadIdx.x & 7, pr = threadIdx.x >> 3;
#pragma unroll
    for (int pp = pr; pp < 64; pp += 32) {
      const int p = p0 + pp, c = c0 + chunk * 8;
      float g8[8], l8[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) g8[i] = l8[i] = 0.f;
      if (p < hw && c < C) {
        const long long o = (static_cast<long long>(b) * V * hw + static_cast<long long>(v) * hw + p) * C + c;
        ld8(dxg + o, g8);
        ld8(dxl + o, l8);
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        tg[pp][chunk * 8 + i] = g8[i];
        tl[pp][chunk * 8 + i] = l8[i];
      }
    }
  }
  __syncthreads();
  float da0 = 0.f, da1 = 0.f;
  if (VEC == 2) {
    const int pl = 2 * tx;
    const float a0 = a_sm[pl], a1 = a_sm[pl + 1];
#pragma unroll
    for (int k = 0; k < 64 / NY; ++k) {
      const int i = ty + k * NY;
      const int c = c0 + i, p = p0 + pl;
      if (c < C && p < hw) {
        const float dl0 = tl[pl][i], dl1 = tl[pl + 1][i];
        st2(df4 + static_cast<long long>(c) * hw + p, tg[pl][i] + a0 * dl0, tg[pl + 1][i] + a1 * dl1);
        da0 = fmaf(fv0[k], dl0, da0);
        da1 = fmaf(fv1[k], dl1, da1);
      }
    }
    da_sm[ty][pl] = da0;
    da_sm[ty][pl + 1] = da1;
  } else {
    const float a = a_sm[tx];
#pragma unroll
    for (int k = 0; k < 64 / NY; ++k) {
      const int i = ty + k * NY;
      const int c = c0 + i, p = p0 + tx;
      if (c < C && p < hw) {
        const float dl = tl[tx][i];
        df4[static_cast<long long>(c) * hw + p] = static_cast<TIO>(tg[tx][i] + a * dl);
        da0 = fmaf(fv0[k], dl, da0);
      }
    }
    da_sm[ty][tx] = da0;
  }
  __syncthreads();
  if (threadIdx.x < 64) {
    const int p = p0 + threadIdx.x;
    if (p < hw) {
      float dA = 0.f;
#pragma unroll
      for (int y = 0; y < NY; ++y) dA += da_sm[y][threadIdx.x];
      da_part[(static_cast<long long>(blockIdx.y) * gridDim.z + bv) * hw + p] = dA;
    }
  }
}

// the chain a = sigmoid(w*m*c), m = sigmoid(max_k cls), c = sigmoid(ctr) backwards for one position
__device__ __forceinline__ void gate_finish_one(const ViewPtrs& vp, int v, int b, int p, int hw, int ncls, float weight,
                                                float a, float dA) {
  const float* cl = vp.cls[v] + static_cast<long long>(b) * ncls * hw + p;
  float lmax = cl[0];
  int arg = 0;
  for (int k = 1; k < ncls; ++k) {
    const float l = cl[static_cast<long long>(k) * hw];
    if (l > lmax) { lmax = l; arg = k; }
  }
  const float m = sigmoidf_(lmax);
  const float c = sigmoidf_(vp.ctr[v][static_cast<long long>(b) * hw + p]);
  const float dt = dA * a * (1.f - a);
  const float dm = dt * weight * c, dc = dt * weight * m;
  vp.dctr[v][static_cast<long long>(b) * hw + p] = dc * c * (1.f - c);
  float* dcl = vp.dcls[v] + static_cast<long long>(b) * ncls * hw + p;
  for (int k = 0; k < ncls; ++k) dcl[static_cast<long long>(k) * hw] = (k == arg) ? dm * m * (1.f - m) : 0.f;
}

// da = sum over channel tiles (fixed order), then the chain a = sigmoid(w*m*c), m = sigmoid(max_k cls), c = sigmoid(ctr)
__global__ void gate_finish_kernel(const ViewPtrs vp, const float* __restrict__ gate, const float* __restrict__ da_part,
                                   int nct, int BV, int V, int hw, int ncls, float weight) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long long>(BV) * hw) return;
  const int bv = static_cast<int>(idx / hw), p = static_cast<int>(idx % hw);
  const int b = bv / V, v = bv % V;
  float dA = 0.f;
  for (int t = 0; t < nct; ++t) dA += da_part[(static_cast<long long>(t) * BV + bv) * hw + p];
  gate_finish_one(vp, v, b, p, hw, ncls, weight, gate[idx], dA);
}

// ------------------------------------------------------------------------------------------------ TMA + ldmatrix forms
// bf16 NCHW views with hw % 8 == 0 and C % 64 == 0 (the cfg2 / network shapes).  One CTA = one (batch, view, 64-position
// block) with ALL channels:
//   * the NCHW side moves as TMA tensor tiles (64 channels x 64 positions, SWIZZLE_128B) and the token-major side as
//     plain bulk copies (64 token rows are one contiguous 64*C*2-byte block), so a CTA has its whole tile (32 KB
//     forward, 96 KB backward) in flight at once — several CTAs per SM keep ~190 KB outstanding;
//   * the 16-bit transposition is done by ldmatrix.trans: with the row -> (channel | position) mapping below a thread
//     receives 8 consecutive channels of one token (forward) or 8 consecutive positions of one channel (backward)
//     as one 16-byte register quad, i.e. exactly one 128-bit global store.
struct ViewMaps {
  CUtensorMap tm[MAXV];
};

__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void bulk_g2s_gate(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

// grid: (ceil(hw/64), B*V); block 256 (8 warps: warp w owns positions 8w..8w+7 of the block).  TIO: bf16 or fp16 f4.
template <typename TIO>
__global__ void __launch_bounds__(256)
    gate_concat_fwd_tma_kernel(const __grid_constant__ ViewMaps maps, const ViewPtrs vp, bf16* __restrict__ xg,
                               bf16* __restrict__ xl, float* __restrict__ gate, int C, int Cs, int V, int hw, int ncls,
                               float weight) {
  // Cs: channels per CTA (a slab of the C channels, blockIdx.z selects it; Cs == C for C <= 512)
  extern __shared__ uint8_t gsm_raw[];
  __shared__ uint64_t bar;
  __shared__ float a_sm[64];
  const uint32_t base = (smem_u32(gsm_raw) + 1023u) & ~1023u;
  const int bv = blockIdx.y, b = bv / V, v = bv % V;
  const int p0 = blockIdx.x * 64;
  const int c_base = blockIdx.z * Cs;
  const int nbox = Cs / 64;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    mbar_init(smem_u32(&bar), 1);
    fence_mbar_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    mbar_expect_tx(smem_u32(&bar), static_cast<uint32_t>(nbox) * 8192u);
    for (int cb = 0; cb < nbox; ++cb)
      tma_load_4d(&maps.tm[v], smem_u32(&bar), base + cb * 8192, p0, c_base + cb * 64, b, 0);
  }
  if (threadIdx.x < 64) {
    const int p = p0 + threadIdx.x;
    float a = 0.f;
    if (p < hw) {
      const float* cl = vp.cls[v] + static_cast<long long>(b) * ncls * hw + p;
      float lmax = cl[0];
      for (int k = 1; k < ncls; ++k) lmax = fmaxf(lmax, cl[static_cast<long long>(k) * hw]);
      const float m = sigmoidf_(lmax);  // max_c sigmoid(l_c) == sigmoid(max_c l_c)
      const float c = sigmoidf_(vp.ctr[v][static_cast<long long>(b) * hw + p]);
      a = sigmoidf_(weight * m * c);
      if (blockIdx.z == 0) gate[static_cast<long long>(bv) * hw + p] = a;
    }
    a_sm[threadIdx.x] = a;
  }
  __syncthreads();
  mbar_wait(smem_u32(&bar), 0);
  // ldmatrix row supplied by this lane: matrix j = lane / 8, row r = lane % 8  <->  channel 8 (r/2) + 2 j + (r%2)
  // of the current 32-channel group; after .trans thread T holds channels 8 (T%4) .. +7 of position T/4
  const int mj = lane >> 3, mr = lane & 7;
  const int co = 8 * (mr >> 1) + 2 * mj + (mr & 1);
  const int pl = warp * 8 + (lane >> 2);          // position of this thread inside the block
  const int p = p0 + pl;
  const float a = a_sm[pl];
  const float2 a2 = make_float2(a, a);
  const long long tok = (static_cast<long long>(b) * V * hw + static_cast<long long>(v) * hw + p) * C + c_base + (lane & 3) * 8;
  const int ngrp = Cs / 32;
#pragma unroll 2
  for (int cg = 0; cg < ngrp; ++cg) {
    const int ch = cg * 32 + co;                  // channel (inside the slab) whose 8-position chunk this lane addresses
    const int row = ch & 63;
    const uint32_t addr = base + (ch >> 6) * 8192 + row * 128 + ((warp ^ (row & 7)) << 4);
    uint32_t r[4];
    ldmatrix_x4_trans(addr, r);
    if (p < hw) {
      uint32_t f[4], g[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 x = unpack2<TIO>(r[i]);
        const float2 y = mul2(x, a2);
        f[i] = std::is_same<TIO, bf16>::value ? r[i] : pack_bf16(x.x, x.y);   // bf16 -> bf16 is the word as it is
        g[i] = pack_bf16(y.x, y.y);
      }
      *reinterpret_cast<uint4*>(xg + tok + cg * 32) = make_uint4(f[0], f[1], f[2], f[3]);
      *reinterpret_cast<uint4*>(xl + tok + cg * 32) = make_uint4(g[0], g[1], g[2], g[3]);
    }
  }
}

// grid: (ceil(hw/64), B*V); block 256.  df4 = dXg + a * dXl back to NCHW and the complete gate gradient
// da[p] = sum_c f4[c,p] * dXl[p,c] (the CTA sees every channel, so no partial table: da_part has one slice).
// TIO: bf16 or fp16 f4 / df4 (the combined gradient is rounded to TIO once, in phase A; phase B moves 16-bit words).
template <typename TIO>
__global__ void __launch_bounds__(256)
    gate_concat_bwd_tma_kernel(const __grid_constant__ ViewMaps maps, const ViewPtrs vp, const float* __restrict__ gate,
                               const bf16* __restrict__ dxg, const bf16* __restrict__ dxl, float* __restrict__ da_part,
                               int Ctot, int C, int V, int hw) {
  // C: channels per CTA (a slab of the Ctot channels, blockIdx.z selects it; C == Ctot for Ctot <= 512): every loop
  // below runs over the slab, only the global addresses know about Ctot; the gate gradient then has one slice per slab
  extern __shared__ uint8_t gsm_raw[];
  __shared__ uint64_t bar;
  __shared__ float a_sm[64];
  const uint32_t base = (smem_u32(gsm_raw) + 1023u) & ~1023u;
  uint8_t* gen = gsm_raw + (base - smem_u32(gsm_raw));
  const int bv = blockIdx.y, b = bv / V, v = bv % V;
  const int p0 = blockIdx.x * 64;
  const int c_base = blockIdx.z * C;
  const int nbox = C / 64;
  const int valid = min(64, hw - p0);
  const uint32_t tile_bytes = 64u * C * 2u;       // one [64 positions][C] bf16 tile
  const uint32_t sF = base, sG = base + tile_bytes, sL = base + 2 * tile_bytes;
  uint8_t* gG = gen + tile_bytes;
  uint8_t* gL = gen + 2 * tile_bytes;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    mbar_init(smem_u32(&bar), 1);
    fence_mbar_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const uint32_t tok_bytes = static_cast<uint32_t>(valid) * C * 2u;
    mbar_expect_tx(smem_u32(&bar), static_cast<uint32_t>(nbox) * 8192u + 2u * tok_bytes);
    for (int cb = 0; cb < nbox; ++cb)
      tma_load_4d(&maps.tm[v], smem_u32(&bar), sF + cb * 8192, p0, c_base + cb * 64, b, 0);
    if (C == Ctot) {               // whole rows: the 64 token rows are one contiguous block
      const long long off = (static_cast<long long>(b) * V * hw + static_cast<long long>(v) * hw + p0) * C;
      bulk_g2s_gate(sG, dxg + off, tok_bytes, smem_u32(&bar));
      bulk_g2s_gate(sL, dxl + off, tok_bytes, smem_u32(&bar));
    }
  }
  if (C != Ctot && static_cast<int>(threadIdx.x) < valid) {     // a slab: one copy per token row and tensor
    const long long off = (static_cast<long long>(b) * V * hw + static_cast<long long>(v) * hw + p0 + threadIdx.x) * Ctot + c_base;
    bulk_g2s_gate(sG + threadIdx.x * C * 2u, dxg + off, static_cast<uint32_t>(C) * 2u, smem_u32(&bar));
    bulk_g2s_gate(sL + threadIdx.x * C * 2u, dxl + off, static_cast<uint32_t>(C) * 2u, smem_u32(&bar));
  }
  if (threadIdx.x < 64) {
    const int p = p0 + threadIdx.x;
    a_sm[threadIdx.x] = p < hw ? gate[static_cast<long long>(bv) * hw + p] : 0.f;
  }
  __syncthreads();
  mbar_wait(smem_u32(&bar), 0);
  const int mj = lane >> 3, mr = lane & 7;
  const int off8 = 8 * (mr >> 1) + 2 * mj + (mr & 1);   // row offset inside a 32-row group addressed by this lane
  const uint32_t row_bytes = static_cast<uint32_t>(C) * 2u;
  {
    // phase A: warp w owns positions 8w..8w+7; per 32-channel group: f4 (transposed through ldmatrix), dXl, dXg ->
    // gate-gradient partial and the combined gradient, written back in place over dXg
    const int pl = warp * 8 + (lane >> 2);
    const float a = a_sm[pl];
    const float2 a2 = make_float2(a, a);
    float2 acc = make_float2(0.f, 0.f);
    const int npair = C / 64;
    const uint32_t rowoff = pl * row_bytes;
    // the combined gradient goes back over dXg with its 16-byte chunks XOR-swizzled by f(pos) (8 distinct values over
    // the 8 rows of a phase-B ldmatrix), which makes the transposing reads of phase B bank-conflict free; the swizzle
    // permutes chunks inside an aligned group of 8 = two 32-channel groups, so both are read before either is written
    const int fsw = ((pl >> 3) & 3) * 2 + (pl & 1);
    for (int cp = 0; cp < npair; ++cp) {
      uint4 gv[2];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int cg = 2 * cp + h;
        const int ch = cg * 32 + off8;
        const int row = ch & 63;
        uint32_t f[4];
        ldmatrix_x4_trans(sF + (ch >> 6) * 8192 + row * 128 + ((warp ^ (row & 7)) << 4), f);
        const uint32_t tokoff = rowoff + (cg * 4 + (lane & 3)) * 16;
        const uint4 lv = *reinterpret_cast<const uint4*>(gL + tokoff);
        gv[h] = *reinterpret_cast<const uint4*>(gG + tokoff);
        const uint32_t* l32 = reinterpret_cast<const uint32_t*>(&lv);
        uint32_t* g32 = reinterpret_cast<uint32_t*>(&gv[h]);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float2 dl = unpack_bf16(l32[i]);
          acc = fma2(unpack2<TIO>(f[i]), dl, acc);
          const float2 t = fma2(a2, dl, unpack_bf16(g32[i]));
          g32[i] = pack2<TIO>(t.x, t.y);
        }
      }
      __syncwarp();
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int c16 = (2 * cp + h) * 4 + (lane & 3);
        *reinterpret_cast<uint4*>(gG + rowoff + ((c16 ^ fsw) << 4)) = gv[h];
      }
      __syncwarp();
    }
    float da = acc.x + acc.y;
    da += __shfl_xor_sync(0xffffffffu, da, 1);
    da += __shfl_xor_sync(0xffffffffu, da, 2);
    if ((lane & 3) == 0 && pl < valid)
      da_part[(static_cast<long long>(blockIdx.z) * gridDim.y + bv) * hw + p0 + pl] = da;
  }
  __syncthreads();
  {
    // phase B: [position][channel] -> NCHW.  ldmatrix rows = positions; thread T receives positions 8 (T%4) .. +7 of
    // channel 8 c8 + T/4
    TIO* df4 = reinterpret_cast<TIO*>(vp.df4[v]) + (static_cast<long long>(b) * Ctot + c_base) * hw;
    const int nunits = 2 * (C / 8);               // (32-position group, 8-channel chunk)
    for (int u = warp; u < nunits; u += 8) {
      const int pg = u & 1, c8 = u >> 1;
      uint32_t r[4];
      const int prow = pg * 32 + off8;
      ldmatrix_x4_trans(sG + prow * row_bytes + ((c8 ^ (((prow >> 3) & 3) * 2 + (prow & 1))) << 4), r);
      const int pp = p0 + pg * 32 + (lane & 3) * 8;
      const int c = c8 * 8 + (lane >> 2);
      if (pp < hw) *reinterpret_cast<uint4*>(df4 + static_cast<long long>(c) * hw + pp) = make_uint4(r[0], r[1], r[2], r[3]);
    }
  }
}

int check_io_dtype(int dt) {
  if (dt == GLF_DTYPE_BF16 || dt == GLF_DTYPE_F16 || dt == GLF_DTYPE_F32) return 0;
  return set_error(GLF_ERR_INVALID, "gate_concat: io_dtype must be GLF_DTYPE_BF16, GLF_DTYPE_F16 or GLF_DTYPE_F32");
}

bool gate_tma_ok(int C, int hw, int io_dtype, int x_dtype, const void* const* f4, int V) {
  if ((io_dtype != GLF_DTYPE_BF16 && io_dtype != GLF_DTYPE_F16) || x_dtype != GLF_DTYPE_BF16) return false;
  if (C % 64 != 0 || hw % 8 != 0) return false;
  if (C > 512 && C % 512 != 0) return false;      // wider rows are cut into 512- (forward) / 256-channel (backward) slabs
  for (int v = 0; v < V; ++v)
    if ((reinterpret_cast<uintptr_t>(f4[v]) & 15) != 0) return false;
  return true;
}

template <typename TX>
int launch_gate_fwd(dim3 grid, bool vec2, int io_dtype, const ViewPtrs& vp, void* xg, void* xl, float* gate, int C, int V,
                    int hw, int ncls, float weight, cudaStream_t stream) {
  if (io_dtype == GLF_DTYPE_BF16) {
    if (vec2) gate_concat_fwd_kernel<bf16, 2, TX><<<grid, 256, 0, stream>>>(vp, (TX*)xg, (TX*)xl, gate, C, V, hw, ncls, weight);
    else gate_concat_fwd_kernel<bf16, 1, TX><<<grid, 256, 0, stream>>>(vp, (TX*)xg, (TX*)xl, gate, C, V, hw, ncls, weight);
  } else if (io_dtype == GLF_DTYPE_F16) {
    if (vec2) gate_concat_fwd_kernel<f16, 2, TX><<<grid, 256, 0, stream>>>(vp, (TX*)xg, (TX*)xl, gate, C, V, hw, ncls, weight);
    else gate_concat_fwd_kernel<f16, 1, TX><<<grid, 256, 0, stream>>>(vp, (TX*)xg, (TX*)xl, gate, C, V, hw, ncls, weight);
  } else {
    if (vec2) gate_concat_fwd_kernel<float, 2, TX><<<grid, 256, 0, stream>>>(vp, (TX*)xg, (TX*)xl, gate, C, V, hw, ncls, weight);
    else gate_concat_fwd_kernel<float, 1, TX><<<grid, 256, 0, stream>>>(vp, (TX*)xg, (TX*)xl, gate, C, V, hw, ncls, weight);
  }
  return check_cuda(cudaGetLastError(), "gate_concat_fwd launch");
}
template <typename TX>
int launch_gate_bwd(dim3 grid, bool vec2, int io_dtype, const ViewPtrs& vp, const float* gate, const void* dxg,
                    const void* dxl, float* da_part, int C, int V, int hw, cudaStream_t stream) {
  if (io_dtype == GLF_DTYPE_BF16) {
    if (vec2) gate_concat_bwd_kernel<bf16, 2, TX><<<grid, 256, 0, stream>>>(vp, gate, (const TX*)dxg, (const TX*)dxl, da_part, C, V, hw);
    else gate_concat_bwd_kernel<bf16, 1, TX><<<grid, 256, 0, stream>>>(vp, gate, (const TX*)dxg, (const TX*)dxl, da_part, C, V, hw);
  } else if (io_dtype == GLF_DTYPE_F16) {
    if (vec2) gate_concat_bwd_kernel<f16, 2, TX><<<grid, 256, 0, stream>>>(vp, gate, (const TX*)dxg, (const TX*)dxl, da_part, C, V, hw);
    else gate_concat_bwd_kernel<f16, 1, TX><<<grid, 256, 0, stream>>>(vp, gate, (const TX*)dxg, (const TX*)dxl, da_part, C, V, hw);
  } else {
    if (vec2) gate_concat_bwd_kernel<float, 2, TX><<<grid, 256, 0, stream>>>(vp, gate, (const TX*)dxg, (const TX*)dxl, da_part, C, V, hw);
    else gate_concat_bwd_kernel<float, 1, TX><<<grid, 256, 0, stream>>>(vp, gate, (const TX*)dxg, (const TX*)dxl, da_part, C, V, hw);
  }
  return check_cuda(cudaGetLastError(), "gate_concat_bwd launch");
}

// ---------------------------------------------------------------------------------------------- channels-last views
// SURVEY.md section 8 f1: when the backbones / heads run channels_last (bf16 autocast), f4[view] arrives as [B, h*w, C]
// rows already - the layout the blocks want - and the NCHW transposition above disappears: gate + concat is a pure row
// kernel (one warp per token, 16-byte accesses along C), and df4 goes back in the same memory format so that the conv
// backward that consumes it stays channels_last.  CL_TOK tokens per warp are kept in flight together.
constexpr int CL_TOK = 4;
struct ClViews {
  const void* f4[MAXV];
  void* df4[MAXV];
  long long sb[MAXV], st[MAXV];       // element strides of batch / token of f4[v]   (channel stride 1)
  long long dsb[MAXV], dst[MAXV];     // ... of df4[v]
};

// raw (still packed) 8-channel vectors: all of a step's loads are issued before the first conversion, and the packed
// form keeps CL_TOK tokens x 3 operands within ~50 registers (the converted form needed 156: one CTA per SM)
template <typename T> struct RawCl;
template <> struct RawCl<bf16> { uint4 v; };
template <> struct RawCl<f16> { uint4 v; };
template <> struct RawCl<float> { float4 a, b; };
__device__ __forceinline__ void ldr(const bf16* p, RawCl<bf16>& r) { r.v = __ldg(reinterpret_cast<const uint4*>(p)); }
__device__ __forceinline__ void ldr(const f16* p, RawCl<f16>& r) { r.v = __ldg(reinterpret_cast<const uint4*>(p)); }
__device__ __forceinline__ void ldr(const float* p, RawCl<float>& r) {
  r.a = __ldg(reinterpret_cast<const float4*>(p));
  r.b = __ldg(reinterpret_cast<const float4*>(p) + 1);
}
__device__ __forceinline__ void cvr(const RawCl<bf16>& r, float (&f)[8]) {
  const uint32_t* u = reinterpret_cast<const uint32_t*>(&r.v);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = unpack_bf16(u[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ void cvr(const RawCl<f16>& r, float (&f)[8]) {
  const uint32_t* u = reinterpret_cast<const uint32_t*>(&r.v);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = unpack2<f16>(u[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ void cvr(const RawCl<float>& r, float (&f)[8]) {
  f[0] = r.a.x; f[1] = r.a.y; f[2] = r.a.z; f[3] = r.a.w;
  f[4] = r.b.x; f[5] = r.b.y; f[6] = r.b.z; f[7] = r.b.w;
}

template <typename TIO>
__global__ void __launch_bounds__(256, 4)
    gate_cl_fwd_kernel(const ClViews cv, const ViewPtrs vp, bf16* __restrict__ xg, bf16* __restrict__ xl,
                       float* __restrict__ gate, int C, int V, int hw, int ncls, float weight) {
  __shared__ float a_sm[8 * CL_TOK];
  const int bv = blockIdx.y, b = bv / V, v = bv % V;
  const int p0 = blockIdx.x * 8 * CL_TOK;
  if (threadIdx.x < 8 * CL_TOK) {
    const int p = p0 + threadIdx.x;
    float a = 0.f;
    if (p < hw) {
      const float* cl = vp.cls[v] + static_cast<long long>(b) * ncls * hw + p;
      float lmax = cl[0];
      for (int k = 1; k < ncls; ++k) lmax = fmaxf(lmax, cl[static_cast<long long>(k) * hw]);
      const float m = sigmoidf_(lmax);
      const float c = sigmoidf_(vp.ctr[v][static_cast<long long>(b) * hw + p]);
      a = sigmoidf_(weight * m * c);
      gate[static_cast<long long>(bv) * hw + p] = a;
    }
    a_sm[threadIdx.x] = a;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const TIO* src = reinterpret_cast<const TIO*>(cv.f4[v]) + b * cv.sb[v];
  const long long st = cv.st[v];
  for (int c = lane * 8; c < C; c += 256) {
    RawCl<TIO> r[CL_TOK];
#pragma unroll
    for (int k = 0; k < CL_TOK; ++k) {
      const int p = p0 + warp * CL_TOK + k;
      if (p < hw) ldr(src + p * st + c, r[k]);
    }
#pragma unroll
    for (int k = 0; k < CL_TOK; ++k) {
      const int p = p0 + warp * CL_TOK + k;
      if (p < hw) {
        const float a = a_sm[warp * CL_TOK + k];
        float f[8], g[8];
        cvr(r[k], f);
#pragma unroll
        for (int i = 0; i < 8; ++i) g[i] = f[i] * a;
        const long long o = (static_cast<long long>(bv) * hw + p) * C + c;
        st8(xg + o, f);
        st8(xl + o, g);
      }
    }
  }
}

template <typename TIO>
__global__ void __launch_bounds__(256, 3)
    gate_cl_bwd_kernel(const ClViews cv, const float* __restrict__ gate, const bf16* __restrict__ dxg,
                       const bf16* __restrict__ dxl, float* __restrict__ da, int C, int V, int hw) {
  const int bv = blockIdx.y, b = bv / V, v = bv % V;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int p0 = blockIdx.x * 8 * CL_TOK + warp * CL_TOK;
  const TIO* src = reinterpret_cast<const TIO*>(cv.f4[v]) + b * cv.sb[v];
  TIO* dst = reinterpret_cast<TIO*>(cv.df4[v]) + b * cv.dsb[v];
  const long long st = cv.st[v], dstt = cv.dst[v];
  float a[CL_TOK], acc[CL_TOK];
#pragma unroll
  for (int k = 0; k < CL_TOK; ++k) {
    a[k] = p0 + k < hw ? gate[static_cast<long long>(bv) * hw + p0 + k] : 0.f;
    acc[k] = 0.f;
  }
  for (int c = lane * 8; c < C; c += 256) {
    RawCl<TIO> rf[CL_TOK];
    RawCl<bf16> rg[CL_TOK], rl[CL_TOK];
#pragma unroll
    for (int k = 0; k < CL_TOK; ++k) {
      const int p = p0 + k;
      if (p < hw) {
        const long long o = (static_cast<long long>(bv) * hw + p) * C + c;
        ldr(src + p * st + c, rf[k]);
        ldr(dxg + o, rg[k]);
        ldr(dxl + o, rl[k]);
      }
    }
#pragma unroll
    for (int k = 0; k < CL_TOK; ++k) {
      const int p = p0 + k;
      if (p < hw) {
        float f[8], g[8], l[8], d[8];
        cvr(rf[k], f);
        cvr(rg[k], g);
        cvr(rl[k], l);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          d[i] = fmaf(a[k], l[i], g[i]);
          acc[k] = fmaf(f[i], l[i], acc[k]);
        }
        st8(dst + p * dstt + c, d);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < CL_TOK; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
    if (lane == 0 && p0 + k < hw) da[static_cast<long long>(bv) * hw + p0 + k] = acc[k];
  }
}

// ---------------------------------------------------------------------------------------------- views -> tokens
// The dict-keyed call site hands the backward one gradient per view ([B, C, h, w], NCHW or channels-last strides);
// the blocks want ONE token-major [B, V, h*w, C] bf16 buffer (the layout ours.py:1819-1820 builds forward).  One
// 64 x 64 tile per CTA; NCHW sources are transposed through shared memory, channels-last sources are row copies.
struct ViewsToTokens {
  const void* src[8];
  long long sb[8], sc[8], st[8];       // element strides of batch / channel / token (= h*w collapsed)
  int present[8];
  int vec[8];                          // channels-last source whose rows can be read 16 bytes at a time
};

template <typename TIn>
__device__ __forceinline__ float ld_as_float(const TIn* p);
template <> __device__ __forceinline__ float ld_as_float<float>(const float* p) { return __ldg(p); }
template <> __device__ __forceinline__ float ld_as_float<bf16>(const bf16* p) { return __bfloat162float(*p); }
template <> __device__ __forceinline__ float ld_as_float<f16>(const f16* p) { return __half2float(*p); }

template <typename TIn>
__global__ void __launch_bounds__(256) views_to_tokens_kernel(ViewsToTokens P, bf16* __restrict__ out, int V, int C,
                                                              int T) {
  __shared__ float tile[64][65];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int tiles_c = C / 64;
  // a CTA owns TWO consecutive 64-token tiles of one 64-channel slab: four 16-byte accesses in flight per thread
  const int tbase = (blockIdx.x / tiles_c) * 128, c0 = (blockIdx.x % tiles_c) * 64;
  const int v = blockIdx.y, b = blockIdx.z;
  bf16* o = out + ((static_cast<long long>(b) * V + v) * T) * C;
  if (!P.present[v]) {                                       // a view without a gradient contributes zeros
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const int t = tbase + ty + 8 * i;
      if (t < T) *reinterpret_cast<__nv_bfloat162*>(o + static_cast<long long>(t) * C + c0 + 2 * tx) = __floats2bfloat162_rn(0.f, 0.f);
    }
    return;
  }
  const TIn* src = reinterpret_cast<const TIn*>(P.src[v]) + b * P.sb[v];
  const long long sc = P.sc[v], st = P.st[v];
  if (sc == 1 && P.vec[v]) {                                 // channels-last rows, 16-byte accesses, loads first
    RawCl<TIn> raw[4];
    int tt[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int item = threadIdx.x + 256 * i;                // 128 tokens x 8 vectors of 8 channels
      tt[i] = tbase + (item >> 3);
      if (tt[i] < T) ldr(src + tt[i] * st + c0 + 8 * (item & 7), raw[i]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (tt[i] < T) {
        bf16* dst = o + static_cast<long long>(tt[i]) * C + c0 + 8 * ((threadIdx.x + 256 * i) & 7);
        if constexpr (std::is_same<TIn, bf16>::value) {
          *reinterpret_cast<uint4*>(dst) = raw[i].v;          // bf16 -> bf16: the packed vector as it is
        } else {
          float f[8];
          cvr(raw[i], f);
          st8(dst, f);
        }
      }
    }
    return;
  }
  for (int half = 0; half < 2; ++half) {
    const int t0 = tbase + 64 * half;
    if (t0 >= T) break;
    if (sc == 1) {                                           // channels-last rows that are not 16-byte aligned
      float lo[8], hi[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int t = t0 + ty + 8 * i;
        const TIn* r = src + t * st + c0 + 2 * tx;
        lo[i] = t < T ? ld_as_float<TIn>(r) : 0.f;
        hi[i] = t < T ? ld_as_float<TIn>(r + 1) : 0.f;
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int t = t0 + ty + 8 * i;
        if (t < T) *reinterpret_cast<__nv_bfloat162*>(o + static_cast<long long>(t) * C + c0 + 2 * tx) = __floats2bfloat162_rn(lo[i], hi[i]);
      }
      continue;
    }
    if (half) __syncthreads();                               // the first half's tile has been read
#pragma unroll
    for (int i = 0; i < 8; ++i) {                            // NCHW: coalesced along tokens, transposed on the way out
      const int c = ty + 8 * i;
      const TIn* r = src + (c0 + c) * sc;
      const int ta = t0 + tx, tb = t0 + 32 + tx;
      tile[c][tx] = ta < T ? ld_as_float<TIn>(r + ta * st) : 0.f;
      tile[c][32 + tx] = tb < T ? ld_as_float<TIn>(r + tb * st) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int tl = ty + 8 * i, t = t0 + tl;
      if (t < T)
        *reinterpret_cast<__nv_bfloat162*>(o + static_cast<long long>(t) * C + c0 + 2 * tx) =
            __floats2bfloat162_rn(tile[2 * tx][tl], tile[2 * tx + 1][tl]);
    }
  }
}

}  // namespace

int views_to_tokens(int B, int C, int V, int T, int src_dtype, const void* const* src, const long long* sb,
                    const long long* sc, const long long* st, void* out, cudaStream_t stream) {
  if (V < 1 || V > 8) return set_error(GLF_ERR_INVALID, "views_to_tokens: V must be 1..8");
  if (C % 64 != 0) return set_error(GLF_ERR_UNSUPPORTED, "views_to_tokens: C %% 64 != 0");
  if (B > 65535) return set_error(GLF_ERR_UNSUPPORTED, "views_to_tokens: B > 65535");
  ViewsToTokens P;
  for (int v = 0; v < 8; ++v) {
    const bool on = v < V && src[v] != nullptr;
    P.src[v] = on ? src[v] : nullptr;
    P.sb[v] = on ? sb[v] : 0; P.sc[v] = on ? sc[v] : 0; P.st[v] = on ? st[v] : 0;
    P.present[v] = on ? 1 : 0;
    const long long per16 = src_dtype == GLF_DTYPE_F32 ? 4 : 8;
    P.vec[v] = on && sc[v] == 1 && reinterpret_cast<uintptr_t>(src[v]) % 16 == 0 && sb[v] % per16 == 0 && st[v] % per16 == 0;
    if (on && sc[v] != 1 && st[v] != 1)
      return set_error(GLF_ERR_UNSUPPORTED, "views_to_tokens: a view needs unit channel or unit token stride");
  }
  const dim3 grid(((T + 127) / 128) * (C / 64), V, B);
  if (src_dtype == GLF_DTYPE_BF16)
    views_to_tokens_kernel<bf16><<<grid, 256, 0, stream>>>(P, reinterpret_cast<bf16*>(out), V, C, T);
  else if (src_dtype == GLF_DTYPE_F16)
    views_to_tokens_kernel<f16><<<grid, 256, 0, stream>>>(P, reinterpret_cast<bf16*>(out), V, C, T);
  else if (src_dtype == GLF_DTYPE_F32)
    views_to_tokens_kernel<float><<<grid, 256, 0, stream>>>(P, reinterpret_cast<bf16*>(out), V, C, T);
  else
    return set_error(GLF_ERR_INVALID, "views_to_tokens: bad dtype");
  return check_cuda(cudaGetLastError(), "views_to_tokens launch");
}

int gate_concat_fwd(int B, int C, int V, int h, int w, int ncls, float weight, int io_dtype, int x_dtype,
                    const void* const* f4, const float* const* cls, const float* const* ctr, void* xg, void* xl,
                    float* gate, cudaStream_t stream) {
  if (V < 1 || V > MAXV) return set_error(GLF_ERR_INVALID, "gate_concat: 1 <= V <= %d", MAXV);
  if (C % 8 != 0) return set_error(GLF_ERR_INVALID, "gate_concat: C %% 8 != 0");
  if (int rc = check_io_dtype(io_dtype)) return rc;
  ViewPtrs vp{};
  for (int v = 0; v < V; ++v) { vp.f4[v] = f4[v]; vp.cls[v] = cls[v]; vp.ctr[v] = ctr[v]; }
  const int hw = h * w;
  if (gate_tma_ok(C, hw, io_dtype, x_dtype, f4, V) && B * V <= 65535) {
    ViewMaps maps;
    for (int v = 0; v < V; ++v) {
      int rc = make_tmap_bf16(&maps.tm[v], f4[v], hw, C, B, hw, static_cast<long long>(C) * hw, 64, io_dtype);
      if (rc) return rc;
    }
    for (int v = V; v < MAXV; ++v) maps.tm[v] = maps.tm[0];
    const int Cs = C <= 512 ? C : 512;
    const uint32_t smem = static_cast<uint32_t>(Cs / 64) * 8192u + 1024u;
    auto kern = io_dtype == GLF_DTYPE_F16 ? gate_concat_fwd_tma_kernel<f16> : gate_concat_fwd_tma_kernel<bf16>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(gate_fwd_tma)");
    kern<<<dim3((hw + 63) / 64, B * V, C / Cs), 256, smem, stream>>>(
        maps, vp, reinterpret_cast<bf16*>(xg), reinterpret_cast<bf16*>(xl), gate, C, Cs, V, hw, ncls, weight);
    return check_cuda(cudaGetLastError(), "gate_concat_fwd_tma launch");
  }
  dim3 grid((hw + 63) / 64, (C + 63) / 64, B * V);
  if (grid.y > 65535 || grid.z > 65535) return set_error(GLF_ERR_INVALID, "gate_concat: grid too large");
  const bool vec2 = (hw % 2 == 0);
  if (x_dtype == GLF_DTYPE_BF16) return launch_gate_fwd<bf16>(grid, vec2, io_dtype, vp, xg, xl, gate, C, V, hw, ncls, weight, stream);
  return launch_gate_fwd<float>(grid, vec2, io_dtype, vp, xg, xl, gate, C, V, hw, ncls, weight, stream);
}

size_t gate_bwd_scratch_bytes(int B, int C, int V, int h, int w) {
  return static_cast<size_t>((C + 63) / 64) * B * V * h * w * sizeof(float);
}

int gate_concat_bwd(int B, int C, int V, int h, int w, int ncls, float weight, int io_dtype, int x_dtype,
                    const void* const* f4, const float* const* cls, const float* const* ctr, const float* gate,
                    const void* dxg, const void* dxl, void* const* df4, float* const* dcls, float* const* dctr,
                    float* da_part, cudaStream_t stream) {
  if (V < 1 || V > MAXV) return set_error(GLF_ERR_INVALID, "gate_concat: 1 <= V <= %d", MAXV);
  if (C % 8 != 0) return set_error(GLF_ERR_INVALID, "gate_concat: C %% 8 != 0");
  if (da_part == nullptr) return set_error(GLF_ERR_WORKSPACE, "gate_concat_bwd: scratch is NULL");
  if (int rc = check_io_dtype(io_dtype)) return rc;
  ViewPtrs vp{};
  for (int v = 0; v < V; ++v) {
    vp.f4[v] = f4[v]; vp.cls[v] = cls[v]; vp.ctr[v] = ctr[v];
    vp.df4[v] = df4[v]; vp.dcls[v] = dcls[v]; vp.dctr[v] = dctr[v];
  }
  const int hw = h * w;
  int nct = (C + 63) / 64;
  bool tma_ok = gate_tma_ok(C, hw, io_dtype, x_dtype, f4, V) && B * V <= 65535 &&
                ((reinterpret_cast<uintptr_t>(dxg) | reinterpret_cast<uintptr_t>(dxl)) & 15) == 0;
  for (int v = 0; v < V && tma_ok; ++v) tma_ok = (reinterpret_cast<uintptr_t>(df4[v]) & 15) == 0;
  if (tma_ok) {
    ViewMaps maps;
    for (int v = 0; v < V; ++v) {
      int rc = make_tmap_bf16(&maps.tm[v], f4[v], hw, C, B, hw, static_cast<long long>(C) * hw, 64, io_dtype);
      if (rc) return rc;
    }
    for (int v = V; v < MAXV; ++v) maps.tm[v] = maps.tm[0];
    const int Cs = C <= 512 ? C : 256;
    const uint32_t smem = 3u * 64u * Cs * 2u + 1024u;
    auto kern = io_dtype == GLF_DTYPE_F16 ? gate_concat_bwd_tma_kernel<f16> : gate_concat_bwd_tma_kernel<bf16>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(gate_bwd_tma)");
    kern<<<dim3((hw + 63) / 64, B * V, C / Cs), 256, smem, stream>>>(
        maps, vp, gate, reinterpret_cast<const bf16*>(dxg), reinterpret_cast<const bf16*>(dxl), da_part, C, Cs, V, hw);
    int rc = check_cuda(cudaGetLastError(), "gate_concat_bwd_tma launch");
    if (rc) return rc;
    // (finishing the chain to the logits inside this kernel was tried: the extra ~2 us at the end of every CTA, two CTAs
    //  per SM and 22 waves, cost 50 us against the 11 us of the launch below)
    nct = C / Cs;   // one slice of the gate-gradient table per channel slab (one for C <= 512)
    const long long n = static_cast<long long>(B) * V * hw;
    gate_finish_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(vp, gate, da_part, nct, B * V, V, hw,
                                                                                  ncls, weight);
    return check_cuda(cudaGetLastError(), "gate_finish launch");
  }
  dim3 grid((hw + 63) / 64, nct, B * V);
  if (grid.y > 65535 || grid.z > 65535) return set_error(GLF_ERR_INVALID, "gate_concat: grid too large");
  const bool vec2 = (hw % 2 == 0);
  int rc = (x_dtype == GLF_DTYPE_BF16)
               ? launch_gate_bwd<bf16>(grid, vec2, io_dtype, vp, gate, dxg, dxl, da_part, C, V, hw, stream)
               : launch_gate_bwd<float>(grid, vec2, io_dtype, vp, gate, dxg, dxl, da_part, C, V, hw, stream);
  if (rc) return rc;
  const long long n = static_cast<long long>(B) * V * hw;
  gate_finish_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(vp, gate, da_part, nct, B * V, V, hw, ncls,
                                                                                weight);
  return check_cuda(cudaGetLastError(), "gate_finish launch");
}

namespace {
int cl_check(int B, int C, int V, int hw, int io_dtype, const void* const* f4, const long long* sb, const long long* st) {
  if (V < 1 || V > MAXV) return set_error(GLF_ERR_INVALID, "gate_concat: 1 <= V <= %d", MAXV);
  if (C % 8 != 0) return set_error(GLF_ERR_INVALID, "gate_concat: C %% 8 != 0");
  if (int rc = check_io_dtype(io_dtype)) return rc;
  if (static_cast<long long>(B) * V > 65535) return set_error(GLF_ERR_UNSUPPORTED, "gate_concat: B * V > 65535");
  const long long per16 = io_dtype == GLF_DTYPE_F32 ? 4 : 8;
  for (int v = 0; v < V; ++v)
    if (f4[v] == nullptr || (reinterpret_cast<uintptr_t>(f4[v]) & 15) != 0 || sb[v] % per16 != 0 || st[v] % per16 != 0 ||
        st[v] < C || (B > 1 && sb[v] < 1))
      return set_error(GLF_ERR_INVALID, "gate_concat (channels-last): view %d needs 16-byte aligned rows of C channels", v);
  (void)hw;
  return 0;
}
}  // namespace

int gate_concat_cl_fwd(int B, int C, int V, int h, int w, int ncls, float weight, int io_dtype, const void* const* f4,
                       const long long* sb, const long long* st, const float* const* cls, const float* const* ctr,
                       void* xg, void* xl, float* gate, cudaStream_t stream) {
  const int hw = h * w;
  int rc = cl_check(B, C, V, hw, io_dtype, f4, sb, st);
  if (rc) return rc;
  ViewPtrs vp{};
  ClViews cv{};
  for (int v = 0; v < V; ++v) {
    vp.cls[v] = cls[v]; vp.ctr[v] = ctr[v];
    cv.f4[v] = f4[v]; cv.sb[v] = sb[v]; cv.st[v] = st[v];
  }
  const dim3 grid((hw + 8 * CL_TOK - 1) / (8 * CL_TOK), B * V);
  if (io_dtype == GLF_DTYPE_BF16)
    gate_cl_fwd_kernel<bf16><<<grid, 256, 0, stream>>>(cv, vp, reinterpret_cast<bf16*>(xg), reinterpret_cast<bf16*>(xl), gate, C, V, hw, ncls, weight);
  else if (io_dtype == GLF_DTYPE_F16)
    gate_cl_fwd_kernel<f16><<<grid, 256, 0, stream>>>(cv, vp, reinterpret_cast<bf16*>(xg), reinterpret_cast<bf16*>(xl), gate, C, V, hw, ncls, weight);
  else
    gate_cl_fwd_kernel<float><<<grid, 256, 0, stream>>>(cv, vp, reinterpret_cast<bf16*>(xg), reinterpret_cast<bf16*>(xl), gate, C, V, hw, ncls, weight);
  return check_cuda(cudaGetLastError(), "gate_cl_fwd launch");
}

int gate_concat_cl_bwd(int B, int C, int V, int h, int w, int ncls, float weight, int io_dtype, const void* const* f4,
                       const long long* sb, const long long* st, const float* const* cls, const float* const* ctr,
                       const float* gate, const void* dxg, const void* dxl, void* const* df4, const long long* dsb,
                       const long long* dst, float* const* dcls, float* const* dctr, float* da, cudaStream_t stream) {
  const int hw = h * w;
  int rc = cl_check(B, C, V, hw, io_dtype, f4, sb, st);
  if (rc) return rc;
  rc = cl_check(B, C, V, hw, io_dtype, df4, dsb, dst);
  if (rc) return rc;
  if (da == nullptr) return set_error(GLF_ERR_WORKSPACE, "gate_concat_bwd: scratch is NULL");
  if (((reinterpret_cast<uintptr_t>(dxg) | reinterpret_cast<uintptr_t>(dxl)) & 15) != 0)
    return set_error(GLF_ERR_INVALID, "gate_concat_bwd: dxg / dxl must be 16-byte aligned");
  ViewPtrs vp{};
  ClViews cv{};
  for (int v = 0; v < V; ++v) {
    vp.cls[v] = cls[v]; vp.ctr[v] = ctr[v]; vp.dcls[v] = dcls[v]; vp.dctr[v] = dctr[v];
    cv.f4[v] = f4[v]; cv.sb[v] = sb[v]; cv.st[v] = st[v];
    cv.df4[v] = df4[v]; cv.dsb[v] = dsb[v]; cv.dst[v] = dst[v];
  }
  const dim3 grid((hw + 8 * CL_TOK - 1) / (8 * CL_TOK), B * V);
  if (io_dtype == GLF_DTYPE_BF16)
    gate_cl_bwd_kernel<bf16><<<grid, 256, 0, stream>>>(cv, gate, reinterpret_cast<const bf16*>(dxg), reinterpret_cast<const bf16*>(dxl), da, C, V, hw);
  else if (io_dtype == GLF_DTYPE_F16)
    gate_cl_bwd_kernel<f16><<<grid, 256, 0, stream>>>(cv, gate, reinterpret_cast<const bf16*>(dxg), reinterpret_cast<const bf16*>(dxl), da, C, V, hw);
  else
    gate_cl_bwd_kernel<float><<<grid, 256, 0, stream>>>(cv, gate, reinterpret_cast<const bf16*>(dxg), reinterpret_cast<const bf16*>(dxl), da, C, V, hw);
  rc = check_cuda(cudaGetLastError(), "gate_cl_bwd launch");
  if (rc) return rc;
  const long long n = static_cast<long long>(B) * V * hw;
  gate_finish_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(vp, gate, da, 1, B * V, V, hw, ncls, weight);
  return check_cuda(cudaGetLastError(), "gate_finish launch");
}

}  // namespace glf
