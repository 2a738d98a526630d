// glf_internal.h — C++ internals shared by the translation units of libglf_sm100a.so.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/glfusion.h"

namespace glf {

int set_error(int code, const char* fmt, ...);   // records thread-local message, returns code
int check_cuda(cudaError_t e, const char* what); // 0 or GLF_ERR_DEVICE
int check_device_sm100();                        // 0 or GLF_ERR_DEVICE

using bf16 = __nv_bfloat16;
using f16 = __half;        // I/O-only element type (GLF_DTYPE_F16): converted to bf16 / fp32 where it is read

#define GLF_TRY(expr)           \
  do {                          \
    int rc__ = (expr);          \
    if (rc__ != 0) return rc__; \
  } while (0)

// Hands out 256-byte aligned pieces of one caller-provided blob in a fixed order; with a NULL base every piece is NULL
// and `off` ends as the blob's size.
struct Carver {
  uint8_t* base;
  size_t off = 0;
  explicit Carver(void* b) : base(reinterpret_cast<uint8_t*>(b)) {}
  template <typename T>
  T* take(size_t n) {
    off = (off + 255) & ~static_cast<size_t>(255);
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += n * sizeof(T);
    return p;
  }
};

// ------------------------------------------------------------------------------------------------ GEMM
struct GemmOperand {
  const void* ptr = nullptr;
  int mn_major = 0;       // 0: [rows, K] K contiguous ; 1: [K, rows] rows contiguous
  int64_t ld = 0;         // leading dimension in elements
  int64_t batch_stride = 0;  // elements; 0 = shared across batch
  int64_t limb_stride = 0;   // elements between bf16 limb planes (F32X3 precision); 0 when single limb
  int rows = 0;              // valid rows of the operand (0 = the GEMM's M / N); smaller values are zero-filled by TMA
};

struct GemmArgs {
  GemmOperand A, B;
  int M = 0, N = 0, K = 0, batch = 1;
  float alpha = 1.f;
  const float* bias = nullptr;      // [N]
  int64_t bias_stride = 0;          // elements between the bias vectors of consecutive batch entries (0 = shared)
  float* rowsum = nullptr;          // optional [batch][M] fp32: sum over K of A's rows (tile N <= 128, npairs == 1);
  int64_t rowsum_stride = 0;        //   stored, or atomically added when split_k > 1 (caller zeroes it then)
  int out_kind = 0;                 // 0 bf16 store, 1 f32 store, 2 f32 atomic add
  void* D = nullptr;
  int64_t ldd = 0, strideD = 0;
  const bf16* addend = nullptr;     // optional bf16 [M, N] added in the epilogue (out_kind 0 only)
  int64_t ld_add = 0, stride_add = 0;
  float* colstats = nullptr;        // partial table, sized for [batch*tiles_m*4][2][N]; rows actually written:
  int* colstats_rows = nullptr;     //   <- returned here (per-CTA running sums shrink it to 4 * gridDim.x rows)
  int split_k = 1;
  int bn_hint = 0;                  // 0 = heuristic, else force the N tile (64 / 128 / 256)
  int npairs = 1;                   // limb products accumulated into one tile: sum_p A[pairA[p]] * B[pairB[p]]^T
  int pairA[6] = {0, 0, 0, 0, 0, 0};
  int pairB[6] = {0, 0, 0, 0, 0, 0};
};
int gemm(const GemmArgs& a, cudaStream_t stream);
inline int gemm_tiles_m(int M) { return (M + 127) / 128; }
inline GemmOperand opnd(const void* p, int mn, long long ld, long long bs, long long limb_stride = 0) {
  GemmOperand o;
  o.ptr = p; o.mn_major = mn; o.ld = ld; o.batch_stride = bs; o.limb_stride = limb_stride;
  return o;
}
// Split-K of a product with `tiles` output tiles and K = `K`
inline int pick_split(long long tiles, int K) {
  const int kb = (K + 63) / 64;
  if (tiles >= 96) return 1;  // enough CTAs already: write the result directly, no atomics
  long long s = (2 * 148) / tiles;   // floor: tiles * s work items fill at most two full rounds of the 148 persistent CTAs
  if (s < 1) s = 1;
  if (s > kb) s = kb;
  return static_cast<int>(s);
}
// (glf_gemm.cu) operand map: K-major -> dims {K, rows, batch, limb}, MN-major -> {rows, K, batch, limb}; SWIZZLE_128B,
// box {64, box_rows or 64}.  Output map: dims {N, M, batch}, box {32, 32}, SWIZZLE_64B (the epilogue's staging tile).
int make_operand_tmap(CUtensorMap* tm, const GemmOperand& op, int rows, int K, int batch, int nlimbs, int box_rows);
int make_output_tmap(CUtensorMap* tm, void* D, int M, int N, int batch, long long ldd, long long strideD);
// (glf_gemm2.cu) the big K-major products with N = 256 on CTA pairs (cta_group::2); false = not applicable / disabled
bool gemm_pair_applicable(const GemmArgs& a, int num_sms);
int gemm_pair(const GemmArgs& a, int num_sms, cudaStream_t stream);
// (glf_gemm3.cu) K-major products with N = 256, K <= 256 whose B operand is shared by many row tiles (U = X Q^T + c per
// sequence): B resident in shared memory, only A streams
bool gemm_bres_applicable(const GemmArgs& a, int num_sms);
int gemm_bres(const GemmArgs& a, int num_sms, cudaStream_t stream);
// (16-bit elements; dtype GLF_DTYPE_BF16 or GLF_DTYPE_F16 names the tensor map's element type)
int make_tmap_bf16(CUtensorMap* tm, const void* ptr, long long inner, long long outer, long long batch, long long ld,
                   long long batch_stride, int box_outer, int dtype = GLF_DTYPE_BF16);

// ------------------------------------------------------------------------------------------------ element-wise
int transpose_cast(const void* in, void* out, int batch, int R, int S, int in_dtype, int out_dtype,
                   cudaStream_t stream);
int prep_weights(const glf_weights* w, int C, int Ci, bf16* wcat, bf16* wcatT, float* bcat, bf16* wz, bf16* wzT,
                 cudaStream_t stream);
// bz: W_z bias that was left out of the stored U (folded into the affine / running mean here), or nullptr
int bn_finalize(const float* part, int np, int C, double count, const glf_desc* d, const glf_weights* w, const float* bz,
                float* mean, float* rstd, float* a, float* b, cudaStream_t stream);
// act_dtype: storage type of the activations U, X (and dV / dU): bf16 in the default path, fp32 under F32X3
int bn_res_ln_fwd(const void* U, const void* X, int act_dtype, const float* a, const float* b, const float* lw,
                  const float* lb, void* Z, int z_dtype, float* mu, float* r, long long rows, int C, float eps,
                  int accumulate, cudaStream_t stream);
int bn_res_ln_bwd_blocks(long long rows, int C);
// *nblocks (optional) receives the number of partial rows written to `part` (<= bn_res_ln_bwd_blocks(rows, C))
int bn_res_ln_bwd(const void* dZ, int dz_dtype, const void* U, const void* X, int act_dtype, const float* a,
                  const float* b, const float* mean, const float* rstd, const float* lw, const float* mu,
                  const float* r, void* dV, float* part, long long rows, int C, int* nblocks, cudaStream_t stream);
// bulk-copy staged forms (glf_ln.cu): bf16 activations, C <= 256; nmod = 2 fuses the MGFM and MLFM LayerNorms.
// Z / Z0 (forward) and dZ / the per-view dz (backward) are of z_dtype: GLF_DTYPE_BF16 or GLF_DTYPE_F16.
bool ln_tma_supported(int C);
int ln_bwd_tma_blocks(long long rows);
int ln_fwd_tma(int nmod, const bf16* const* U, const bf16* const* X, const float* const* a, const float* const* b,
               const float* const* lw, const float* const* lb, float* const* mu, float* const* r, void* Z,
               long long rows, int C, float eps, int accumulate, cudaStream_t stream, void* Z0 = nullptr,
               int z_dtype = GLF_DTYPE_BF16);
int ln_bwd_tma(int nmod, const void* dZ, const bf16* const* U, const bf16* const* X, const float* const* a,
               const float* const* b, const float* const* lw, const float* const* bn_mean,
               const float* const* bn_rstd, const float* const* mu, const float* const* r, bf16* const* dV,
               float* const* part, long long rows, int C, int* nblocks, cudaStream_t stream, int dz_nv = 0,
               const void* const* dz_views = nullptr, const long long* dz_sb = nullptr, int dz_hw = 0,
               int dz_dtype = GLF_DTYPE_BF16);
int ln_bwd_tma_tile_rows();
// (glf_eltwise.cu) the fused MGFM + MLFM LayerNorm forward for wide rows, 256 < C <= 2048 (sliced rows, cp.async ring)
bool ln_pair_wide_supported(int C);
int ln_pair_fwd_wide(const bf16* const* U, const bf16* const* X, const float* const* a, const float* const* b,
                     const float* const* lw, const float* const* lb, float* const* mu, float* const* r, void* Z,
                     long long rows, int C, float eps, int accumulate, cudaStream_t stream, void* Z0,
                     int z_dtype = GLF_DTYPE_BF16);
int bn_bwd_finalize(const float* part, int np, int C, double count, const glf_desc* d, const glf_weights* w,
                    const float* mean, const float* rstd, const glf_grads* g, float* k1, float* k2, float* k3,
                    cudaStream_t stream);
int bn_bwd_apply(const void* dV, const void* U, int act_dtype, const float* k1, const float* k2, const float* k3,
                 void* dU, long long rows, int C, cudaStream_t stream);
int split3(const float* in, bf16* out, long long n, cudaStream_t stream);   // fp32 [n] -> bf16 limbs [3][n]
int colstats_f32_blocks(long long rows);
int colstats_f32(const float* A, float* part, long long rows, int C, cudaStream_t stream);
int prep_weights_f32(const glf_weights* w, int C, int Ci, float* wcat, float* wcatT, float* bcat, cudaStream_t stream);
// Two-stage reductions: stage 1 shrinks a table of `np` partial rows to REDUCE_STAGE1_ROWS rows (parallel, fixed order).
constexpr int REDUCE_STAGE1_ROWS = 64;
int reduce_stage1(const float* p0, const float* p1, const float* p2, int ntab, const int* np_in, int* np,
                  long long* row_stride, long long stat_stride, int NS, int C, float* scratch, cudaStream_t stream);
int reduce_partials(const float* part, int np, long long stride, int n, float alpha, float* out, cudaStream_t stream);
int reduce_partials3(const float* p0, const float* p1, const float* p2, int np, long long stride, int n, float* o0,
                     float* o1, float* o2, cudaStream_t stream);
int cast_bf16(const float* in, bf16* out, long long n, cudaStream_t stream);
// GLF_DTYPE_* element type of the glf_weights / glf_grads tensors (glf_desc.reserved[3], validated by make_dims)
inline int param_dtype(const glf_desc* d) {
  return d->reserved[3] == GLF_PARAMS_BF16 ? GLF_DTYPE_BF16 : d->reserved[3] == GLF_PARAMS_F16 ? GLF_DTYPE_F16 : GLF_DTYPE_F32;
}
// A block's twelve parameter tensors (glf_grads order) copied between two element types in one launch: 2-byte
// masters -> fp32 (forward) or fp32 gradients -> 2-byte, rounded to nearest (backward).  A NULL src or dst is skipped.
constexpr int NPARAMS = 12;
struct ParamCopy {
  const void* src[NPARAMS];
  void* dst[NPARAMS];
  long long n[NPARAMS];
};
int convert_params(const ParamCopy& p, int src_dtype, int dst_dtype, cudaStream_t stream);

// ------------------------------------------------------------------------------------------------ Gram form (glf_gram.cu)
// Augmented width of the per-sequence matrices: column C is the homogeneous coordinate, the rest zero padding.
inline int gram_ca(int C) { return C + 8; }
int gram_prep_weights(const glf_weights* w, int C, int Ci, int Ca, bf16* waug, bf16* wzb, cudaStream_t stream);
// the same conversion as extra CTAs of the S contraction's launch (gram_kernel): no launch of its own
struct GramPrep {
  const float *tw, *tb, *pw, *pb, *gw, *gb, *wz;
  bf16 *waug, *wzb;
  int C, Ci, Ca;
};
// rowscale (optional, [C]): rows < C of the augmented matrix (column C included) are scaled per row
int gram_assemble_aug(const float* Mf, const float* colv, const float* rowv, const float* rowscale, bf16* out, int B,
                      int C, int Ca, float corner, cudaStream_t stream);
int gram_border(const float* colv, const float* rowv, const float* rowscale, bf16* out, int B, int C, int Ca,
                float corner, cudaStream_t stream);
int gram_cvec(const bf16* Wp, const float* theta_b, float* cvec, int B, int C, int Ci, cudaStream_t stream);
int gram_kprep(const bf16* Qb, const float* cvec, const float* k1, const float* k2, const float* k3, bf16* AK, bf16* EF,
               int B, int C, int Ca, cudaStream_t stream);
int gram_assemble_F(const bf16* G0, const bf16* Hf, const bf16* dT, const bf16* wphi, bf16* EF, float* evec, int B,
                    int C, int Ci, int Ca, cudaStream_t stream);
// One CTA per sequence (glf_gramk.cu): D_b = A_b^T X_b for C = 128 / 256, operands streamed once
bool gram_contraction_supported(int C);
int gram_contraction(const bf16* A, const bf16* X, bf16* out_aug, float* scratch, float* rowsum, const float* rowscale,
                     const float* rowv, float corner, int border, int B, int N, int C, int Ca, int ksplit,
                     cudaStream_t stream, const GramPrep* prep = nullptr);
int gram_unpack_grads(const float* dwaug, const glf_grads* g, int C, int Ci, int Ca, cudaStream_t stream);
// One CTA per sequence runs the whole [C x C] chain between the token-sized products (glf_chain.cu), C = 256, C' = 128
bool gram_chain_supported(int C, int Ci);
int gram_chain_fwd(const bf16* Sa, const float* sfv, const bf16* waug, const bf16* wz, const float* bphi,
                   const float* bg, const float* bth, bf16* T, bf16* Mb, bf16* Wp, bf16* Qb, float* cvec, float* tv, int B,
                   int N, cudaStream_t stream);
// dMn = dM / N.  has_k2 = 0 skips the Q^T (k2 Q) term (k2 = k3 = 0: eval-mode BatchNorm or bn_layer = False)
int gram_chain_bwd(const bf16* Sa, const bf16* Qb, const bf16* waug, const bf16* wz, const bf16* Rb, const float* sfv,
                   const float* cvec, const float* rv, const float* k1, const float* k2, const float* k3,
                   const float* bth, const float* bphi, const float* bg, int has_k2, bf16* dQa, bf16* dWp, bf16* dMn,
                   bf16* dT, bf16* EF, float* evec, float* dcv, float* dtv, int B, int N, cudaStream_t stream);
// The four weight-gradient sums over the sequences as ONE launch of K-concatenated products + a fixed-order reduction
// of the per-CTA partials (glf_wgrad.cu); writes theta / phi / g weight + bias gradients and wz_w.
size_t gram_wgrad_scratch_floats();
int gram_wgrad(const bf16* Wp, const bf16* dQa, const bf16* dWp, const bf16* Mb, const bf16* dMn, const bf16* T,
               const bf16* dT, const bf16* Sa, const float* dcv, const float* tv, const float* dtv, const float* sfv,
               float* part, const glf_grads* g, int B, int N, cudaStream_t stream);

// ------------------------------------------------------------------------------------------------ gate + concat
int gate_concat_fwd(int B, int C, int V, int h, int w, int ncls, float weight, int io_dtype, int x_dtype,
                    const void* const* f4, const float* const* cls, const float* const* ctr, void* xg, void* xl,
                    float* gate, cudaStream_t stream);
int gate_concat_bwd(int B, int C, int V, int h, int w, int ncls, float weight, int io_dtype, int x_dtype,
                    const void* const* f4, const float* const* cls, const float* const* ctr, const float* gate,
                    const void* dxg, const void* dxl, void* const* df4, float* const* dcls, float* const* dctr,
                    float* da_part, cudaStream_t stream);
size_t gate_bwd_scratch_bytes(int B, int C, int V, int h, int w);
// channels-last views (element (b, c, t) at b*sb + t*st + c): gate + concat / its backward as row kernels; df4 in the
// layout given by dsb / dst; da: [B*V*h*w] floats of scratch (gate_bwd_scratch_bytes covers it)
int gate_concat_cl_fwd(int B, int C, int V, int h, int w, int ncls, float weight, int io_dtype, const void* const* f4,
                       const long long* sb, const long long* st, const float* const* cls, const float* const* ctr,
                       void* xg, void* xl, float* gate, cudaStream_t stream);
int gate_concat_cl_bwd(int B, int C, int V, int h, int w, int ncls, float weight, int io_dtype, const void* const* f4,
                       const long long* sb, const long long* st, const float* const* cls, const float* const* ctr,
                       const float* gate, const void* dxg, const void* dxl, void* const* df4, const long long* dsb,
                       const long long* dst, float* const* dcls, float* const* dctr, float* da, cudaStream_t stream);
// per-view [B,C,h,w] tensors (element strides sb / sc / st of batch, channel, collapsed h*w) -> token-major
// [B, V, T, C] bf16; a NULL view is written as zeros
int views_to_tokens(int B, int C, int V, int T, int src_dtype, const void* const* src, const long long* sb,
                    const long long* sc, const long long* st, void* out, cudaStream_t stream);

// ------------------------------------------------------------------------------------------------ cycle step
// (glf_cycle.cu) the consumer of the MGFM output: per-view spatial sums (R/main.py:229) and the cycle-consistency
// loss with its gradient (R/main.py:650-798), n_starts start positions start, start+step, ...
size_t cycle_loss_scratch_bytes(int T, int C, int n_starts);
int cycle_loss(const float* feat, int T, int C, int R, int off, int ch, float temperature, int start, int step,
               int n_starts, int soft_label, float scale, float* loss, float* dfeat, float* scratch,
               cudaStream_t stream);
int spatial_sums(const void* x, int dtype, int B, int C, int T, long long sb, long long sc, long long st, float* out,
                 cudaStream_t stream);

// ------------------------------------------------------------------------------------------------ softmax attention
// mode='embedded' (ours.py:896-897,902): Y = softmax(Theta Phi^T) G, flash-style, per batch entry;
// mode='gaussian' (ours.py:869-873): Y = softmax(X X^T) G.
// P: [B, N, 3Ci] bf16 (theta | phi | g); Y: [B, N, Ci] bf16; lse: [B, N] fp32 (natural-log-sum-exp per query row)
int attn_ld(int N);
int attn_chunk(long long B, long long N);
size_t attn_scratch_bytes(long long B, long long N, bool backward);
int flash_fwd(const bf16* P, bf16* Y, float* lse, int B, int N, int Ci, void* scratch, cudaStream_t stream);
// Partial column sums of the outputs that carry a bias: table i holds rows[i] rows of [2][width] floats at tab[i] (the
// sums first), consecutive rows `stride` floats apart in every table of the set.
struct ColTables {
  int n = 0;
  const float* tab[3] = {nullptr, nullptr, nullptr};
  int rows[3] = {0, 0, 0};
  long long stride = 0;
};
// cs: the column sums of dP = [dTheta | dPhi | dG], three tables
int flash_bwd(const bf16* P, const bf16* Y, const bf16* dY, const float* lse, bf16* dP, float* delta, float* cs_t,
              float* cs_p, float* cs_g, int cs_cap_rows, ColTables* cs, int B, int N, int Ci, void* scratch,
              cudaStream_t stream);
// The same attention with Q, K and V given separately: Y = softmax(Q K^T) V per sequence, Q / K of width wqk, V / Y / dY
// of width wv, every operand token rows with its own leading dimension.  mode='embedded' is Q = Theta, K = Phi, V = G
// (slots of one [Theta | Phi | G] row); mode='gaussian' (ours.py:869-873) is Q = K = X (wqk = C) and V = G (wv = C').
// Flash kernels for (wqk, wv) in {(64, 64), (128, 64), (128, 128)}, the chunked exact path otherwise.
struct AttnArgs {
  const bf16 *q = nullptr, *k = nullptr, *v = nullptr;
  long long ldq = 0, ldk = 0, ldv = 0;
  int wqk = 0, wv = 0;
  bf16 *dq = nullptr, *dk = nullptr, *dvo = nullptr;    // backward outputs dQ, dK, dV (no atomics: each is stored once)
  long long ld_dq = 0, ld_dk = 0, ld_dv = 0;
  bool bias_qkv = true;   // bias sums over [dQ | dK | dV] (adjacent slots of one row, 'embedded'), else over dV alone
};
AttnArgs attn_args_embedded(const bf16* P3, bf16* dP3, int Ci);
AttnArgs attn_args_gaussian(const bf16* X, const bf16* G, bf16* dXa, bf16* dXb, bf16* dG, long long ld_dx,
                            long long ld_dg, int C, int Ci);
bool attn_flash_supported(int wqk, int wv);
int attn_fwd(const AttnArgs& a, bf16* Y, float* lse, int B, int N, void* scratch, cudaStream_t stream);
// cs: the column sums of [dQ | dK | dV] (bias_qkv, three tables) or of dV alone (one table), written into the
// cs_t / cs_p / cs_g scratch (cs_cap_rows rows of [2][width] each)
int attn_bwd(const AttnArgs& a, const bf16* Y, const bf16* dY, const float* lse, float* delta, float* cs_t, float* cs_p,
             float* cs_g, int cs_cap_rows, ColTables* cs, int B, int N, void* scratch, cudaStream_t stream);
// out [rows, C] = in[:, :C] + in[:, C:2C] for in [rows, 2C] bf16 (fp32 sum, rounded once)
int sum_halves(const bf16* in, bf16* out, long long rows, int C, cudaStream_t stream);
// mode='gaussian' weights: wg [Ci, C] = bf16(g.weight), bg [Ci] = g.bias, wgT [C, 2C + Ci] = [I | I | g.weight^T] (the dX
// product's B operand: dX = [dS X | dS^T X | dG] wgT^T), wz [C, Ci], wzT [Ci, C]
int prep_weights_gaussian(const glf_weights* w, int C, int Ci, bf16* wg, bf16* wgT, float* bg, bf16* wz, bf16* wzT,
                          cudaStream_t stream);

// ------------------------------------------------------------------------------------------------ P2P all-reduce (glf_p2p.cu)
int p2p_grid(long long n_floats);
long long p2p_max_floats();
size_t p2p_signal_bytes(int world);
int p2p_allreduce(void* const* bufs, void* const* sigs, int rank, int world, long long n_floats, float scale,
                  cudaStream_t stream);
int p2p_export(const void* ptr, unsigned char handle[64], unsigned long long* offset);
int p2p_open(const unsigned char handle[64], unsigned long long offset, void** out);
int p2p_close(void* ptr, unsigned long long offset);

// ------------------------------------------------------------------------------------------------ TPAVIModule (glf_api.cu)
// One block's problem, validated and derived from its glf_desc by make_dims.
struct Dims {
  long long B, N, rows;
  int C, Ci;
  int tiles_seq;   // m-tiles per sequence (128 tokens)
  int tiles_all;   // m-tiles over all rows
  bool pack_x;     // x must be repacked to token-major in the working dtype (bf16, or fp32 under F32X3)
  bool pack_dz;
  bool dot;
  bool gauss;      // mode='gaussian': Q = K = X, only the g projection runs
  bool gram;       // mode='dot' in its Gram form (channel-space products only)
  int Ca;          // augmented width of the per-sequence matrices (gram)
  int pdt;         // GLF_DTYPE_* of the glf_weights / glf_grads tensors (glf_desc.reserved[3])
  bool half_params;   // bf16 / fp16 parameters: an fp32 shadow in `saved`, fp32 gradient staging in ws_bwd
};
// x / dz (in_dtype, [B, C, N] when ncthw, else token-major) -> token-major [B * N, C] of out_dtype;
// unpack_tokens is the way back for dx
int pack_tokens(const Dims& m, const void* in, int in_dtype, bool ncthw, void* out, int out_dtype, cudaStream_t stream);
int unpack_tokens(const Dims& m, const void* in, int in_dtype, void* out, bool ncthw, int out_dtype,
                  cudaStream_t stream);
// dWcat = [dtheta_w ; dphi_w ; dg_w] (Ci x C each), or dg_w alone (g_only), into the gradient tensors
int scatter_proj_grads(const float* dwcat, const glf_grads* g, int C, int Ci, bool g_only, cudaStream_t stream);

// ------------------------------------------------------------------------------------------------ F32X3 precision arm
int tpavi_sizes_f32x3(const glf_desc* d, const Dims& m, glf_sizes* out);
int tpavi_fwd_f32x3(const glf_desc* d, const Dims& m, const void* x, const glf_weights* w, void* z, void* saved,
                    void* ws, cudaStream_t stream);
int tpavi_bwd_f32x3(const glf_desc* d, const Dims& m, const void* dz, const void* x, const glf_weights* w,
                    const void* saved, void* dx, const glf_grads* g, void* ws, cudaStream_t stream);

}  // namespace glf
