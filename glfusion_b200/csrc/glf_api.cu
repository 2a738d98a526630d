// glf_api.cu — the C ABI (include/glfusion.h) and the host-side orchestration of one TPAVIModule forward/backward
// (R/models/ours.py:845-917) as a fixed sequence of kernel launches on the caller's stream.  No allocation, no
// synchronisation: the whole sequence is CUDA-graph capturable.
//
// mode='dot' is executed in its reassociated O(N C'^2) form (SURVEY.md F2), token-major throughout:
//   fwd:  P=[Theta|Phi|G] = X Wcat^T + b         tcgen05 GEMM (x read once, three projections concatenated)
//         M_b = Phi_b^T G_b / N                   tcgen05 GEMM, MN-major operands, split-K, fp32 red.add
//         W'_b = W_z M_b^T                        small fp32 SIMT product (C x C' per sequence)
//         U_b = Theta_b W'_b^T + b_z              tcgen05 GEMM + per-tile BatchNorm column statistics
//         BN finalise, then  Z = LN(BN(U) + X)    HBM-bound fused epilogue
//   bwd:  LN/BN backward (two HBM-bound passes), then six tcgen05 GEMMs (dTheta, dW', dPhi, dG, dWcat, dX) and two
//         small fp32 products (dW_z, dM).
// mode='embedded' and mode='gaussian' run the softmax attention of glf_flash.cu between the projection and the W_z GEMM;
// gaussian projects g alone (P = G) and its attention reads x itself as Q and K, so dX gets dS X + dS^T X as well.
// When the sequences are long against the channel count (N >= 5 C) mode='dot' runs in its Gram form instead
// (tpavi_fwd_gram / tpavi_bwd_gram below; oracle/tpavi_oracle.py: tpavi_dot_gram_form): theta / phi / g and dU are never
// materialised, the only token-sized products are S = X^T X, U = X Q^T, R = dV^T X and dX = [dV | X] [E ; F].
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "glf_internal.h"

namespace glf {

static thread_local char g_err[512] = "";

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
int check_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return 0;
  return set_error(GLF_ERR_DEVICE, "%s: %s", what, cudaGetErrorString(e));
}
int check_device_sm100() {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return check_cuda(e, "cudaGetDevice");
  int major = 0, minor = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
  if (major != 10) return set_error(GLF_ERR_DEVICE, "libglf_sm100a needs an sm_100 device (Blackwell B200); found sm_%d%d and there is no fallback path", major, minor);
  return 0;
}

int pack_tokens(const Dims& m, const void* in, int in_dtype, bool ncthw, void* out, int out_dtype, cudaStream_t stream) {
  if (ncthw)
    return transpose_cast(in, out, static_cast<int>(m.B), m.C, static_cast<int>(m.N), in_dtype, out_dtype, stream);
  return transpose_cast(in, out, 1, 1, static_cast<int>(m.rows * m.C), in_dtype, out_dtype, stream);   // cast only
}

int unpack_tokens(const Dims& m, const void* in, int in_dtype, void* out, bool ncthw, int out_dtype,
                  cudaStream_t stream) {
  if (ncthw)
    return transpose_cast(in, out, static_cast<int>(m.B), static_cast<int>(m.N), m.C, in_dtype, out_dtype, stream);
  return transpose_cast(in, out, 1, 1, static_cast<int>(m.rows * m.C), in_dtype, out_dtype, stream);
}

int scatter_proj_grads(const float* dwcat, const glf_grads* g, int C, int Ci, bool g_only, cudaStream_t stream) {
  float* const dst[3] = {g->theta_w, g->phi_w, g->g_w};
  const char* what[3] = {"copy dtheta", "copy dphi", "copy dg"};
  const size_t n = static_cast<size_t>(Ci) * C;
  for (int k = g_only ? 2 : 0, row = 0; k < 3; ++k, ++row)
    GLF_TRY(check_cuda(cudaMemcpyAsync(dst[k], dwcat + row * n, sizeof(float) * n, cudaMemcpyDeviceToDevice, stream),
                       what[k]));
  return 0;
}

namespace {

int make_dims(const glf_desc* d, Dims* o) {
  if (d == nullptr) return set_error(GLF_ERR_INVALID, "null descriptor");
  if (d->B <= 0 || d->T <= 0 || d->H <= 0 || d->W <= 0) return set_error(GLF_ERR_INVALID, "empty input (B,T,H,W must be > 0)");
  if (d->C <= 0 || d->Ci <= 0 || d->C % 8 != 0 || d->Ci % 8 != 0)
    return set_error(GLF_ERR_INVALID, "C and inter_channels must be positive multiples of 8 (got %d, %d)", d->C, d->Ci);
  if (d->C > 2048) return set_error(GLF_ERR_INVALID, "C <= 2048 supported (got %d)", d->C);
  if (d->mode != GLF_MODE_DOT && d->mode != GLF_MODE_EMBEDDED && d->mode != GLF_MODE_GAUSSIAN)
    return set_error(GLF_ERR_UNSUPPORTED, "mode must be dot, embedded or gaussian ('concatenate' is not built by the reference network)");
  if (d->precision != GLF_PRECISION_BF16 && d->precision != GLF_PRECISION_F32X3)
    return set_error(GLF_ERR_INVALID, "bad precision (GLF_PRECISION_BF16 or GLF_PRECISION_F32X3)");
  if (d->precision == GLF_PRECISION_F32X3 && d->mode != GLF_MODE_DOT)
    return set_error(GLF_ERR_UNSUPPORTED, "GLF_PRECISION_F32X3 is implemented for mode='dot' only");
  if (d->io_dtype != GLF_DTYPE_BF16 && d->io_dtype != GLF_DTYPE_F32 && d->io_dtype != GLF_DTYPE_F16)
    return set_error(GLF_ERR_INVALID, "bad io_dtype (GLF_DTYPE_BF16, GLF_DTYPE_F32 or GLF_DTYPE_F16)");
  // the exact arm is an fp32 contract: fp16 inputs (11-bit significands, 65504 range) would defeat it
  if (d->precision == GLF_PRECISION_F32X3 && d->io_dtype == GLF_DTYPE_F16)
    return set_error(GLF_ERR_UNSUPPORTED, "GLF_PRECISION_F32X3 takes fp32 or bf16 activations, not fp16 (GLF_DTYPE_F16)");
  if (d->reserved[2] != GLF_DTYPE_BF16 && d->reserved[2] != GLF_DTYPE_F16)
    return set_error(GLF_ERR_INVALID, "reserved[2] (dtype of the fused LayerNorm's z / dz) must be GLF_DTYPE_BF16 or GLF_DTYPE_F16");
  if (d->reserved[3] != GLF_PARAMS_F32 && d->reserved[3] != GLF_PARAMS_BF16 && d->reserved[3] != GLF_PARAMS_F16)
    return set_error(GLF_ERR_INVALID, "reserved[3] (parameter dtype) must be GLF_PARAMS_F32, GLF_PARAMS_BF16 or GLF_PARAMS_F16");
  // the exact arm is an fp32 contract for the parameters too
  if (d->precision == GLF_PRECISION_F32X3 && d->reserved[3] != GLF_PARAMS_F32)
    return set_error(GLF_ERR_UNSUPPORTED, "GLF_PRECISION_F32X3 takes fp32 parameters, not bf16 / fp16 (reserved[3])");
  o->pdt = param_dtype(d);
  o->half_params = o->pdt != GLF_DTYPE_F32;
  o->B = d->B;
  o->N = static_cast<long long>(d->T) * d->H * d->W;
  o->rows = o->B * o->N;
  if (o->rows * static_cast<long long>(d->C) >= (1LL << 40)) return set_error(GLF_ERR_INVALID, "problem too large");
  if (o->N > (1LL << 30)) return set_error(GLF_ERR_INVALID, "sequence too long");
  o->C = d->C;
  o->Ci = d->Ci;
  o->tiles_seq = gemm_tiles_m(static_cast<int>(o->N));
  o->tiles_all = gemm_tiles_m(static_cast<int>(o->rows > 0x7fffffff ? 0x7fffffff : o->rows));
  if (o->rows > 0x7fffff00LL) return set_error(GLF_ERR_INVALID, "too many tokens");
  const int work_dtype = d->precision == GLF_PRECISION_F32X3 ? GLF_DTYPE_F32 : GLF_DTYPE_BF16;
  o->pack_x = !(d->x_layout == GLF_LAYOUT_TOKEN && d->io_dtype == work_dtype);
  if (d->x_layout == GLF_LAYOUT_TOKEN && d->io_dtype != GLF_DTYPE_BF16 && o->rows * d->C > 0x7fffffffLL)
    return set_error(GLF_ERR_INVALID, "token-major fp32 / fp16 input too large for the cast kernel");
  o->pack_dz = d->dz_layout != GLF_LAYOUT_TOKEN;
  o->dot = d->mode == GLF_MODE_DOT;
  o->gauss = d->mode == GLF_MODE_GAUSSIAN;
  // reserved[1]: 0 = choose, 1 = token-space form (theta/phi/g per token), 2 = Gram form; | GLF_DETERMINISTIC
  const int algo = d->reserved[1] & 0xff, flags = d->reserved[1] & ~0xff;
  if (algo > 2 || (flags != 0 && flags != GLF_DETERMINISTIC))
    return set_error(GLF_ERR_INVALID, "reserved[1] must be the dot algorithm 0, 1 or 2, optionally ORed with "
                                      "GLF_DETERMINISTIC (0x100) (got 0x%x)", static_cast<unsigned>(d->reserved[1]));
  o->det = flags == GLF_DETERMINISTIC;
  const bool gram_ok = o->dot && d->precision == GLF_PRECISION_BF16 && o->B <= 65535;
  if (algo == 2 && !gram_ok)
    return set_error(GLF_ERR_UNSUPPORTED, "the Gram form needs mode='dot', GLF_PRECISION_BF16 and B <= 65535");
  // per-sequence [C x C] products cost ~15 C^3 against 3.5 N C^2 of saved token-space FLOPs and 11 saved activation
  // passes.  Measured crossover on B200 (profiles/algo_crossover.py, r02_algo_crossover.txt): with the one-CTA-per-
  // sequence chain kernels (C = 256, C' = 128) the Gram form wins from N/C = 3 (1.00 vs 1.11 ms at N = 784, B = 512);
  // at C = 128 between 3 and 24; above C = 256 the token-space form (every GEMM on CTA pairs) still wins at N/C = 6
  // (C = 512: 1.37 vs 1.46 ms; C = 1024: 1.85 vs 1.96 ms).
  const long long thr = gram_chain_supported(d->C, d->Ci) ? 3 : (d->C > 256 ? 8 : 5);
  o->gram = gram_ok && (algo == 2 || (algo == 0 && o->N >= thr * d->C));
  o->Ca = gram_ca(d->C);
  return 0;
}

// Element counts of the twelve parameter tensors, glf_grads order.
void param_counts(const Dims& m, long long n[NPARAMS]) {
  const long long CCi = static_cast<long long>(m.C) * m.Ci;
  const long long v[NPARAMS] = {CCi, m.Ci, CCi, m.Ci, CCi, m.Ci, CCi, m.C, m.C, m.C, m.C, m.C};
  for (int k = 0; k < NPARAMS; ++k) n[k] = v[k];
}
// fp32 copies of the twelve parameter tensors (half parameters only; NULL otherwise)
void carve_params(Carver& c, const Dims& m, float* out[NPARAMS]) {
  long long n[NPARAMS];
  param_counts(m, n);
  for (int k = 0; k < NPARAMS; ++k) out[k] = m.half_params ? c.take<float>(n[k]) : nullptr;
}
void weight_list(const glf_weights* w, const void* p[NPARAMS]) {
  const void* v[NPARAMS] = {w->theta_w, w->theta_b, w->phi_w, w->phi_b, w->g_w, w->g_b,
                            w->wz_w,    w->wz_b,    w->bn_w,  w->bn_b,  w->ln_w, w->ln_b};
  for (int k = 0; k < NPARAMS; ++k) p[k] = v[k];
}
// The parameters every kernel reads: the caller's tensors, or with bf16 / fp16 parameters their fp32 shadow `sh`
// (running statistics untouched: bn_finalize reads and updates them in their own dtype); an absent tensor (bn_layer = 0)
// stays absent
glf_weights fp32_weights(const Dims& m, const glf_weights* w, float* const sh[NPARAMS]) {
  glf_weights o = *w;
  if (!m.half_params) return o;
  const float** f[NPARAMS] = {&o.theta_w, &o.theta_b, &o.phi_w, &o.phi_b, &o.g_w, &o.g_b,
                              &o.wz_w,    &o.wz_b,    &o.bn_w,  &o.bn_b,  &o.ln_w, &o.ln_b};
  for (int k = 0; k < NPARAMS; ++k) *f[k] = *f[k] != nullptr ? sh[k] : nullptr;
  return o;
}
// The gradient targets every writer fills: the caller's tensors, or with bf16 / fp16 parameters the fp32 staging `st`
// that emit_grads rounds into them
glf_grads fp32_grads(const Dims& m, const glf_grads* g, float* const st[NPARAMS]) {
  if (!m.half_params) return *g;
  glf_grads o;
  float** f[NPARAMS] = {&o.theta_w, &o.theta_b, &o.phi_w, &o.phi_b, &o.g_w, &o.g_b,
                        &o.wz_w,    &o.wz_b,    &o.bn_w,  &o.bn_b,  &o.ln_w, &o.ln_b};
  for (int k = 0; k < NPARAMS; ++k) *f[k] = st[k];
  return o;
}
// forward: the 2-byte masters into the fp32 shadow that every consumer reads
int stage_params(const Dims& m, const glf_weights* w, float* const sh[NPARAMS], cudaStream_t stream) {
  ParamCopy p;
  weight_list(w, p.src);
  param_counts(m, p.n);
  for (int k = 0; k < NPARAMS; ++k) p.dst[k] = sh[k];
  return convert_params(p, m.pdt, GLF_DTYPE_F32, stream);
}
// backward: the fp32 gradients every writer left in the staging area, rounded into the caller's tensors
int emit_grads(const Dims& m, float* const st[NPARAMS], const glf_grads* g, cudaStream_t stream) {
  if (!m.half_params) return 0;
  ParamCopy p;
  void* v[NPARAMS] = {g->theta_w, g->theta_b, g->phi_w, g->phi_b, g->g_w, g->g_b,
                      g->wz_w,    g->wz_b,    g->bn_w,  g->bn_b,  g->ln_w, g->ln_b};
  param_counts(m, p.n);
  for (int k = 0; k < NPARAMS; ++k) {
    p.src[k] = st[k];
    p.dst[k] = (m.gauss && k < 4) ? nullptr : v[k];   // gaussian: theta / phi take no part and receive no gradient
  }
  return convert_params(p, GLF_DTYPE_F32, m.pdt, stream);
}

struct Saved {
  float* pshadow[NPARAMS];    // fp32 copies of bf16 / fp16 parameters (the fused LayerNorm pass reads ln_w / ln_b here)
  bf16 *xtok, *P, *Y, *U, *Mb, *Wp, *wcat, *wcatT, *wz, *wzT;
  float *lse, *bcat, *bn_mean, *bn_rstd, *bn_a, *bn_b, *ln_mu, *ln_r;
  bf16 *Sa, *T, *Qb, *waug;   // Gram form: S~ [B][Ca][Ca], T = W~phi S~ [B][Ci][Ca], Q~ [B][C][Ca], W~ [3][Ci][Ca]
  float *sfv, *cvec;          //            s = column sums of X [B][C], c = Q~[:, :, C] [B][C]
  float *tv;                  //            t = T~[:, :, C] [B][Ci] in fp32 (chain kernels)
};
size_t carve_saved(const Dims& m, void* base, Saved* s) {
  Carver c(base);
  const size_t rows = m.rows, C = m.C, Ci = m.Ci, B = m.B;
  carve_params(c, m, s->pshadow);
  s->xtok = m.pack_x ? c.take<bf16>(rows * C) : nullptr;
  s->Sa = s->T = s->Qb = s->waug = nullptr;
  s->sfv = s->cvec = s->tv = nullptr;
  if (m.gram) {
    const size_t Ca = m.Ca;
    s->P = s->Y = s->wcat = s->wcatT = s->wzT = nullptr;
    s->lse = s->bcat = nullptr;
    s->U = c.take<bf16>(rows * C);
    s->Sa = c.take<bf16>(B * Ca * Ca);
    s->T = c.take<bf16>(B * Ci * Ca);
    s->Mb = c.take<bf16>(B * Ci * Ci);
    s->Wp = c.take<bf16>(B * C * Ci);
    s->Qb = c.take<bf16>(B * C * Ca);
    s->waug = c.take<bf16>(3 * Ci * Ca);
    s->wz = c.take<bf16>(C * Ci);
    s->sfv = c.take<float>(B * C);
    s->cvec = c.take<float>(B * C);
    s->tv = c.take<float>(B * Ci);
    s->bn_mean = c.take<float>(C);
    s->bn_rstd = c.take<float>(C);
    s->bn_a = c.take<float>(C);
    s->bn_b = c.take<float>(C);
    s->ln_mu = c.take<float>(rows);
    s->ln_r = c.take<float>(rows);
    return (c.off + 255) & ~static_cast<size_t>(255);
  }
  s->P = c.take<bf16>(rows * (m.gauss ? Ci : 3 * Ci));   // [Theta | Phi | G], or G alone (gaussian)
  s->U = c.take<bf16>(rows * C);
  if (m.dot) {
    s->Y = nullptr; s->lse = nullptr;
    s->Mb = c.take<bf16>(B * Ci * Ci);
    s->Wp = c.take<bf16>(B * C * Ci);
  } else {
    s->Y = c.take<bf16>(rows * Ci);
    s->lse = c.take<float>(rows);
    s->Mb = nullptr; s->Wp = nullptr;
  }
  // gaussian: wcat = W_g [Ci, C], bcat = b_g, wcatT = [I | I | W_g^T] [C, 2C + Ci] (prep_weights_gaussian)
  s->wcat = c.take<bf16>((m.gauss ? 1 : 3) * Ci * C);
  s->wcatT = c.take<bf16>(m.gauss ? C * (2 * C + Ci) : 3 * Ci * C);
  s->bcat = c.take<float>((m.gauss ? 1 : 3) * Ci);
  s->wz = c.take<bf16>(C * Ci);
  s->wzT = c.take<bf16>(C * Ci);
  s->bn_mean = c.take<float>(C);
  s->bn_rstd = c.take<float>(C);
  s->bn_a = c.take<float>(C);
  s->bn_b = c.take<float>(C);
  s->ln_mu = c.take<float>(rows);
  s->ln_r = c.take<float>(rows);
  return (c.off + 255) & ~static_cast<size_t>(255);
}

// The two blocks' operands of the fused LayerNorm pass (index 0 = MGFM, 1 = MLFM) from their saved blobs, with ln_w /
// ln_b as the kernels read them (the fp32 shadow of bf16 / fp16 parameters)
struct LnPair {
  const bf16 *U[2], *X[2];
  const float *a[2], *b[2], *mean[2], *rstd[2], *lw[2], *lb[2];
  float *mu[2], *r[2];
};
LnPair ln_pair(const Dims& m, const void* xg, const void* xl, const glf_weights* wg, const glf_weights* wl,
               const void* saved_g, const void* saved_l) {
  const void* x[2] = {xg, xl};
  const glf_weights* w[2] = {wg, wl};
  const void* saved[2] = {saved_g, saved_l};
  LnPair p;
  for (int k = 0; k < 2; ++k) {
    Saved s;
    carve_saved(m, const_cast<void*>(saved[k]), &s);
    const glf_weights w32 = fp32_weights(m, w[k], s.pshadow);
    p.U[k] = s.U;
    p.X[k] = reinterpret_cast<const bf16*>(x[k]);
    p.a[k] = s.bn_a; p.b[k] = s.bn_b; p.mean[k] = s.bn_mean; p.rstd[k] = s.bn_rstd;
    p.lw[k] = w32.ln_w; p.lb[k] = w32.ln_b;
    p.mu[k] = s.ln_mu; p.r[k] = s.ln_r;
  }
  return p;
}

int pick_split_rounds(long long M, long long N, long long batch, int K);
// K slices of the one-CTA-per-sequence token contraction: few long sequences are split to fill two rounds of the SMs
int gram_ksplit(long long B) { return B < 96 ? ((2 * 148) / B < 1 ? 1 : static_cast<int>((2 * 148) / B)) : 1; }

// Slab floats of the fixed-order split reductions (GLF_DETERMINISTIC): the largest need among the products of the
// forward (or backward) that sum partials, with the splits those products pick
long long det_slab_floats(const Dims& m, bool backward) {
  const int B = static_cast<int>(m.B), C = m.C, Ci = m.Ci, N = static_cast<int>(m.N), rows = static_cast<int>(m.rows);
  auto t = [](long long n) { return (n + 127) / 128; };
  long long need = 0;
  auto take = [&need](long long v) { need = v > need ? v : need; };
  if (m.gram) {   // S = X^T X forward, R = dV^T X backward: the same shapes
    if (gram_contraction_supported(C)) take(gram_slab_floats(B, N, C, gram_ksplit(B)));
    else take(slab_need(C, C, B, N, pick_split(B * t(C) * t(C), N), false, true));
    if (backward && !gram_chain_supported(C, Ci)) {   // dW~theta / dW~phi / dW~g and dWz summed over the sequences
      take(slab_need(Ci, m.Ca, B, C, 1, true, false));
      take(slab_need(C, Ci, B, Ci, 1, true, false));
    }
    return need;
  }
  if (m.dot) {
    if (!backward) take(slab_need(Ci, Ci, B, N, pick_split(B * t(Ci) * t(Ci), N), false, false));     // M
    else {
      take(slab_need(C, Ci, B, N, pick_split(B * t(C) * t(Ci), N), false, false));                    // dW'
      take(slab_need(C, Ci, B, Ci, 1, true, false));                                                  // dWz
    }
  } else if (backward) {
    take(slab_need(C, Ci, 1, rows, pick_split_rounds(C, Ci, 1, rows), false, false));                 // dWz
  }
  if (backward) {
    const int nproj = m.gauss ? Ci : 3 * Ci;
    take(slab_need(nproj, C, 1, rows, pick_split_rounds(nproj, C, 1, rows), false, false));           // dWcat
  }
  return need;
}
// The slabs go last in ws, so that every other piece keeps its offset whether the flag is set or not
void carve_slab(Carver& c, const Dims& m, bool backward, SplitSlab* s) {
  *s = SplitSlab{};
  if (!m.det) return;
  s->on = true;
  s->floats = det_slab_floats(m, backward);
  if (s->floats > 0) s->p = c.take<float>(static_cast<size_t>(s->floats));
}

struct WsFwd { float* colstats; float* red1; float* Mf; void* attn; void* saved_fallback; float* Sf; SplitSlab det; };
size_t carve_ws_fwd(const Dims& m, void* base, WsFwd* w, size_t saved_bytes) {
  Carver c(base);
  const size_t np = 4 * (m.dot ? static_cast<size_t>(m.B) * m.tiles_seq : static_cast<size_t>(m.tiles_all));
  w->colstats = c.take<float>(np * 2 * m.C);   // one partial per (tile, 32-row quarter)
  w->red1 = c.take<float>(static_cast<size_t>(REDUCE_STAGE1_ROWS) * 2 * m.C);
  w->Sf = nullptr;
  if (m.gram) {
    w->Mf = nullptr; w->attn = nullptr;
    w->Sf = c.take<float>(static_cast<size_t>(m.B) * m.C * m.C);   // split-K accumulation target of S = X^T X
    w->saved_fallback = c.take<uint8_t>(saved_bytes);
    carve_slab(c, m, false, &w->det);
    return (c.off + 255) & ~static_cast<size_t>(255);
  }
  w->Mf = m.dot ? c.take<float>(static_cast<size_t>(m.B) * m.Ci * m.Ci) : nullptr;  // split-K accumulation target
  w->attn = m.dot ? nullptr : c.take<uint8_t>(attn_scratch_bytes(m.B, m.N, false));
  w->saved_fallback = c.take<uint8_t>(saved_bytes);  // used when the caller passes saved == NULL (inference)
  carve_slab(c, m, false, &w->det);
  return (c.off + 255) & ~static_cast<size_t>(255);
}

struct WsBwd {
  float* gstage[NPARAMS];     // fp32 gradients of bf16 / fp16 parameters, before emit_grads rounds them
  bf16 *dztok, *dV, *dU, *dP, *dY, *dxtok, *dM, *dWpb;
  float *dWpf, *part_ln, *k1, *k2, *k3, *cs_t, *cs_p, *cs_g, *red1, *dwcat, *delta;
  void* attn;
  // Gram form
  float *Rf, *rv, *evec, *dwaug, *dcv, *dtv, *wpart;
  bf16 *Rb, *AK, *dQa, *dT, *EF, *G0, *Hf;
  SplitSlab det;
};
size_t carve_ws_bwd(const glf_desc* d, const Dims& m, void* base, WsBwd* w) {
  Carver c(base);
  const size_t rows = m.rows, C = m.C, Ci = m.Ci, B = m.B;
  carve_params(c, m, w->gstage);
  w->dztok = m.pack_dz ? c.take<bf16>(rows * C) : nullptr;
  w->dV = c.take<bf16>(rows * C);
  w->Rf = w->rv = w->evec = w->dwaug = w->dcv = w->dtv = w->wpart = nullptr;
  w->Rb = w->AK = w->dQa = w->dT = w->EF = w->G0 = w->Hf = nullptr;
  if (m.gram) {
    const size_t Ca = m.Ca;
    w->dU = w->dP = w->dY = nullptr;
    w->dWpf = w->cs_t = w->cs_p = w->cs_g = w->red1 = w->dwcat = w->delta = nullptr;
    w->attn = nullptr;
    w->dxtok = m.pack_x ? c.take<bf16>(rows * C) : nullptr;
    w->part_ln = c.take<float>(static_cast<size_t>(bn_res_ln_bwd_blocks(m.rows, m.C)) * 4 * C);
    w->k1 = c.take<float>(C);
    w->k2 = c.take<float>(C);
    w->k3 = c.take<float>(C);
    w->Rf = c.take<float>(B * C * C);        // split-K accumulation target of R = dV^T X
    w->rv = c.take<float>(B * C);
    w->Rb = c.take<bf16>(B * Ca * Ca);       // k1 [R | rv] (rows < C)
    w->AK = c.take<bf16>(B * C * Ca);        // Qk = k2 Q~ (column C: k2 c + k3) per sequence
    w->dQa = c.take<bf16>(B * C * Ca);
    w->dWpb = c.take<bf16>(B * C * Ci);
    w->dM = c.take<bf16>(B * Ci * Ci);
    w->dT = c.take<bf16>(B * Ci * Ca);
    w->G0 = c.take<bf16>(B * C * Ca);        // dS~[:C, :] (the three terms of F are rounded to bf16, summed in fp32)
    w->Hf = c.take<bf16>(B * C * Ca);
    w->EF = c.take<bf16>(B * 2 * C * C);
    w->evec = c.take<float>(B * C);
    w->dwaug = c.take<float>(3 * Ci * Ca);
    w->dcv = c.take<float>(B * C);
    w->dtv = c.take<float>(B * Ci);
    w->wpart = gram_chain_supported(m.C, m.Ci) ? c.take<float>(gram_wgrad_scratch_floats()) : nullptr;
    carve_slab(c, m, true, &w->det);
    return (c.off + 255) & ~static_cast<size_t>(255);
  }
  w->dU = d->bn_layer ? c.take<bf16>(rows * C) : nullptr;
  w->dP = c.take<bf16>(rows * (m.gauss ? 2 * C + Ci : 3 * Ci));   // [dTheta | dPhi | dG], or [dS X | dS^T X | dG]
  w->dxtok = m.pack_x ? c.take<bf16>(rows * C) : nullptr;
  if (m.dot) {
    w->dY = nullptr; w->delta = nullptr;
    w->dWpf = c.take<float>(B * C * Ci);
    w->dWpb = c.take<bf16>(B * C * Ci);
    w->dM = c.take<bf16>(B * Ci * Ci);
  } else {
    w->dY = c.take<bf16>(rows * Ci);
    w->delta = c.take<float>(rows);
    w->dWpf = nullptr; w->dWpb = nullptr; w->dM = nullptr;
  }
  w->attn = m.dot ? nullptr : c.take<uint8_t>(attn_scratch_bytes(m.B, m.N, true));
  w->part_ln = c.take<float>(static_cast<size_t>(bn_res_ln_bwd_blocks(m.rows, m.C)) * 4 * C);
  w->k1 = c.take<float>(C);
  w->k2 = c.take<float>(C);
  w->k3 = c.take<float>(C);
  const size_t np = 4 * B * m.tiles_seq;       // one partial per (tile, 32-row quarter)
  w->cs_t = c.take<float>(np * 2 * Ci);
  w->cs_p = c.take<float>(np * 2 * Ci);
  w->cs_g = c.take<float>(np * 2 * Ci);
  w->red1 = c.take<float>(static_cast<size_t>(REDUCE_STAGE1_ROWS) * 3 * Ci);
  w->dwcat = c.take<float>(3 * Ci * C);
  carve_slab(c, m, true, &w->det);
  return (c.off + 255) & ~static_cast<size_t>(255);
}

// A per-sequence token contraction (K = N) of the token-space form into bf16 D [batch][M][N]: written directly when
// there are enough output tiles, else split along K with fp32 red.add into `acc` (zeroed first), rounded once into D.
int token_contraction(GemmArgs g, bf16* D, float* acc, cudaStream_t stream) {
  const long long n = static_cast<long long>(g.batch) * g.M * g.N;
  g.ldd = g.N; g.strideD = static_cast<long long>(g.M) * g.N;
  g.split_k = pick_split(static_cast<long long>(g.batch) * ((g.M + 127) / 128) * ((g.N + 127) / 128), g.K);
  if (g.split_k == 1) {
    g.out_kind = 0;
    g.D = D;
    return gemm(g, stream);
  }
  GLF_TRY(check_cuda(cudaMemsetAsync(acc, 0, sizeof(float) * n, stream), "memset split-K accumulator"));
  g.out_kind = 2;
  g.D = acc;
  GLF_TRY(gemm(g, stream));
  return cast_bf16(acc, D, n, stream);
}

// Split of a long token contraction (K = all rows) whose output tiles alone leave the last round of the 148 persistent
// CTAs mostly empty: e.g. dWcat at C = 2048 is 24 x 8 = 192 tiles of 128 x 256 = 1.3 rounds (0.65 of the machine);
// three K-slices make 576 work items = 3.9 rounds of a third the length (0.97).  Mirrors gemm()'s tile choice.
int pick_split_rounds(long long M, long long N, long long batch, int K) {
  const long long BNt = N <= 64 ? 64 : ((K >= 512 && N % 256 == 0) ? 256 : 128);
  const long long tiles = ((M + 127) / 128) * ((N + BNt - 1) / BNt) * batch;
  if (tiles < 96) return pick_split(tiles, K);
  const int kb = (K + 63) / 64;
  int best = 1;
  double best_eff = 0.0;
  for (int sp = 1; sp <= 4 && kb / sp >= 16; ++sp) {
    const long long items = tiles * sp;
    const double eff = static_cast<double>(items) / (148.0 * static_cast<double>((items + 147) / 148));
    if (eff > best_eff + 0.08) { best_eff = eff; best = sp; }     // a further slice has to buy 8 % of the machine
  }
  return best;
}

// reserved[0] = 1: the LayerNorm stage (forward epilogue / first backward kernel) is run for MGFM and MLFM together
// by glf_fusion_ln_fwd / glf_fusion_ln_bwd instead of per block
bool defer_ln(const glf_desc* d) { return d->reserved[0] == 1; }
// reserved[2]: dtype of z / z_global / dz of the fused LayerNorm pass (make_dims admits GLF_DTYPE_BF16 = 0 or F16)
int pair_z_dtype(const glf_desc* d) { return d->reserved[2]; }

int check_pair(const glf_desc* d, const Dims& m) {
  if (d->precision != GLF_PRECISION_BF16 || d->io_dtype != GLF_DTYPE_BF16 || m.pack_x || d->dz_layout != GLF_LAYOUT_TOKEN)
    return set_error(GLF_ERR_UNSUPPORTED, "fused LayerNorm pair needs bf16 token-major x_g / x_l and token-major dz");
  if (!ln_tma_supported(m.C) && !ln_pair_wide_supported(m.C))
    return set_error(GLF_ERR_UNSUPPORTED, "fused LayerNorm pair needs C %% 8 == 0 and C <= 2048");
  return 0;
}

int check_ptr(const void* p, const char* name) {
  if (p == nullptr) return set_error(GLF_ERR_INVALID, "%s is NULL", name);
  if ((reinterpret_cast<uintptr_t>(p) & 15) != 0) return set_error(GLF_ERR_INVALID, "%s must be 16-byte aligned", name);
  return 0;
}


// ------------------------------------------------------------------------------------------------ Gram form of 'dot'
// The Ca-wide small products and U / dX run on 128-wide N tiles (bn_hint = 128). Measured on B200 at cfg2
// (profiles/README.md): 128 is faster than the 256-wide tile, which has only three ring stages for four k-blocks per
// tile and which gemm()'s heuristic would pick for U and dX at C >= 512.

// Token contraction of a sequence, S = A^T X (A = X or dV): both operands MN-major views of token-major
// activations, the column sums of A as the GEMM's row-sum side product; result = the augmented bf16 matrix
// [[S, colsum(A)], [rowv^T, corner]] of width Ca.  Enough sequences: the GEMM writes bf16 straight into it and a border
// kernel adds the homogeneous row / column; few long sequences: split-K into fp32, then one assembling pass.
int gram_token_contraction(const bf16* A, const bf16* X, bf16* out_aug, float* scratch, float* rowsum, const float* rowv,
                           const float* rowscale, float corner, int B, int N, int C, int Ca, const SplitSlab& det,
                           cudaStream_t stream, const GramPrep* prep = nullptr, bool* prep_done = nullptr) {
  if (prep_done != nullptr) *prep_done = false;
  if (gram_contraction_supported(C)) {
    // one CTA per sequence; few long sequences are split along the tokens to fill two rounds of the SMs
    const int ks = gram_ksplit(B);
    GLF_TRY(gram_contraction(A, X, out_aug, scratch, rowsum, rowscale, rowv, corner, 1, B, N, C, Ca, ks, stream, prep,
                             &det));
    if (prep != nullptr && prep_done != nullptr) *prep_done = true;
    const int kb = (N + 63) / 64;
    if ((ks > kb ? kb : ks) > 1)
      return gram_assemble_aug(scratch, rowsum, rowv ? rowv : rowsum, rowscale, out_aug, B, C, Ca, corner, stream);
    return 0;   // one CTA per sequence: the kernel wrote the border as well
  }
  GemmArgs g;
  g.A = opnd(A, 1, C, static_cast<long long>(N) * C);
  g.B = opnd(X, 1, C, static_cast<long long>(N) * C);
  g.M = C; g.N = C; g.K = N; g.batch = B;
  g.bn_hint = 128;
  g.rowsum = rowsum; g.rowsum_stride = C;
  g.det = det;
  g.split_k = pick_split(static_cast<long long>(B) * ((C + 127) / 128) * ((C + 127) / 128), N);
  if (g.split_k > 1 || rowscale != nullptr) {   // (a per-row scale needs the fp32 result: the GEMM's alpha is a scalar)
    if (g.split_k > 1) {
      GLF_TRY(check_cuda(cudaMemsetAsync(scratch, 0, sizeof(float) * B * C * C, stream), "memset S"));
      GLF_TRY(check_cuda(cudaMemsetAsync(rowsum, 0, sizeof(float) * B * C, stream), "memset s"));
    }
    g.out_kind = g.split_k > 1 ? 2 : 1;
    g.D = scratch; g.ldd = C; g.strideD = static_cast<long long>(C) * C;
    GLF_TRY(gemm(g, stream));
    return gram_assemble_aug(scratch, rowsum, rowv ? rowv : rowsum, rowscale, out_aug, B, C, Ca, corner, stream);
  }
  g.out_kind = 0;
  g.D = out_aug; g.ldd = Ca; g.strideD = static_cast<long long>(Ca) * Ca;
  GLF_TRY(gemm(g, stream));
  return gram_border(rowsum, rowv ? rowv : rowsum, nullptr, out_aug, B, C, Ca, corner, stream);
}

// D = A0 B0^T + A1 B1^T (+ bias + addend), bf16 output: both products accumulate into one TMEM tile when each operand
// pair can be described as two "limbs" of one tensor map (their distance in memory is the limb stride); otherwise two
// passes, the second adding onto the first in place.  g.A / g.B carry layout, leading dimension and batch stride.
int gemm_pair2(GemmArgs g, const bf16* A0, const bf16* A1, const bf16* B0, const bf16* B1, cudaStream_t stream) {
  const long long dA = A1 - A0, dB = B1 - B0;
  auto ok = [](long long d) {
    const long long a = d < 0 ? -d : d;
    return a != 0 && a % 8 == 0 && a < (1LL << 38);
  };
  if (ok(dA) && ok(dB)) {
    g.A.ptr = dA > 0 ? A0 : A1; g.A.limb_stride = dA > 0 ? dA : -dA;
    g.B.ptr = dB > 0 ? B0 : B1; g.B.limb_stride = dB > 0 ? dB : -dB;
    g.npairs = 2;
    g.pairA[0] = dA > 0 ? 0 : 1; g.pairA[1] = 1 - g.pairA[0];
    g.pairB[0] = dB > 0 ? 0 : 1; g.pairB[1] = 1 - g.pairB[0];
    return gemm(g, stream);
  }
  g.A.ptr = A0; g.B.ptr = B0;
  GLF_TRY(gemm(g, stream));
  g.A.ptr = A1; g.B.ptr = B1;
  g.bias = nullptr;
  g.addend = reinterpret_cast<const bf16*>(g.D); g.ld_add = g.ldd; g.stride_add = g.strideD;
  return gemm(g, stream);
}

// The end of the forward from the U product on: its np rows of BatchNorm column statistics (shrunk by a stage-1
// reduction when long) finalised into the affine, then Z = LN(BN(U) + X) unless the fused LayerNorm pair
// (glf_fusion_ln_fwd) finishes both blocks in one pass
int bn_ln_fwd(const glf_desc* d, const Dims& m, const bf16* X, const glf_weights* w, int np, void* z, const Saved& s,
              const WsFwd& wf, cudaStream_t stream) {
  const int C = m.C;
  const float* bn_part = wf.colstats;
  if (d->training && d->bn_layer && np > 4 * REDUCE_STAGE1_ROWS) {
    long long rs = 2LL * C;
    const int np_in[1] = {np};
    GLF_TRY(reduce_stage1(wf.colstats, nullptr, nullptr, 1, np_in, &np, &rs, C, 2, C, wf.red1, stream));
    bn_part = wf.red1;
  }
  GLF_TRY(bn_finalize(bn_part, np, C, static_cast<double>(m.rows), d, w, w->wz_b, s.bn_mean, s.bn_rstd, s.bn_a, s.bn_b,
                      stream));
  if (defer_ln(d)) return 0;
  GLF_TRY(bn_res_ln_fwd(s.U, X, GLF_DTYPE_BF16, s.bn_a, s.bn_b, w->ln_w, w->ln_b, z, d->io_dtype, s.ln_mu, s.ln_r,
                        m.rows, C, d->eps_ln, d->accumulate, stream));
  return 0;
}

int tpavi_fwd_gram(const glf_desc* d, const Dims& m, const void* x, const glf_weights* w, void* z, const Saved& s,
                   const WsFwd& wf, cudaStream_t stream) {
  const int C = m.C, Ci = m.Ci, Ca = m.Ca, C1 = m.C + 1;
  const int N = static_cast<int>(m.N), B = static_cast<int>(m.B);
  const long long CaCa = static_cast<long long>(Ca) * Ca, CiCa = static_cast<long long>(Ci) * Ca;
  const long long CCa = static_cast<long long>(C) * Ca, CiCi = static_cast<long long>(Ci) * Ci;
  const long long CCi = static_cast<long long>(C) * Ci;
  const bf16* X = reinterpret_cast<const bf16*>(x);
  if (m.pack_x) {
    GLF_TRY(pack_tokens(m, x, d->io_dtype, d->x_layout == GLF_LAYOUT_NCTHW, s.xtok, GLF_DTYPE_BF16, stream));
    X = s.xtok;
  }
  // S_b = X_b^T X_b, s_b = X_b^T 1   ->   S~_b
  //   (the fp32 -> bf16 weight preparation for the chain that follows rides along as extra CTAs of the same launch)
  GramPrep prep;
  prep.tw = w->theta_w; prep.tb = w->theta_b; prep.pw = w->phi_w; prep.pb = w->phi_b; prep.gw = w->g_w; prep.gb = w->g_b;
  prep.wz = w->wz_w; prep.waug = s.waug; prep.wzb = s.wz; prep.C = C; prep.Ci = Ci; prep.Ca = Ca;
  bool prep_done = false;
  GLF_TRY(gram_token_contraction(X, X, s.Sa, wf.Sf, s.sfv, nullptr, nullptr, static_cast<float>(N), B, N, C, Ca, wf.det,
                                 stream, &prep, &prep_done));
  if (!prep_done) GLF_TRY(gram_prep_weights(w, C, Ci, Ca, s.waug, s.wz, stream));
  if (gram_chain_supported(C, Ci)) {
    // T~, M, W', Q~ and c of every sequence in one launch, one CTA per sequence (glf_chain.cu)
    GLF_TRY(gram_chain_fwd(s.Sa, s.sfv, s.waug, s.wz, w->phi_b, w->g_b, w->theta_b, s.T, s.Mb, s.Wp, s.Qb, s.cvec, s.tv, B,
                           N, stream));
  } else {
    {  // T_b = W~phi S~_b                      [Ci x Ca]   (= Phi_b^T X~_b; S~ is symmetric)
      GemmArgs g;
      g.A = opnd(s.waug + CiCa, 0, Ca, 0);
      g.B = opnd(s.Sa, 0, Ca, CaCa);
      g.B.rows = C1;
      g.M = Ci; g.N = Ca; g.K = C1; g.batch = B;
      g.bn_hint = 128;
      g.D = s.T; g.ldd = Ca; g.strideD = CiCa;
      GLF_TRY(gemm(g, stream));
    }
    {  // M_b = T_b W~g^T / N                   [Ci x Ci]   (= Phi_b^T G_b / N)
      GemmArgs g;
      g.A = opnd(s.T, 0, Ca, CiCa);
      g.B = opnd(s.waug + 2 * CiCa, 0, Ca, 0);
      g.M = Ci; g.N = Ci; g.K = C1; g.batch = B;
      g.alpha = 1.f / static_cast<float>(N);
      g.D = s.Mb; g.ldd = Ci; g.strideD = CiCi;
      GLF_TRY(gemm(g, stream));
    }
    {  // W'_b = Wz M_b^T                       [C x Ci]
      GemmArgs g;
      g.A = opnd(s.wz, 0, Ci, 0);
      g.B = opnd(s.Mb, 0, Ci, CiCi);
      g.M = C; g.N = Ci; g.K = Ci; g.batch = B;
      g.D = s.Wp; g.ldd = Ci; g.strideD = CCi;
      GLF_TRY(gemm(g, stream));
    }
    {  // Q~_b = W'_b W~theta                   [C x Ca]    (B operand = W~theta read MN-major: stored [K = i][rows = a])
      GemmArgs g;
      g.A = opnd(s.Wp, 0, Ci, CCi);
      g.B = opnd(s.waug, 1, Ca, 0);
      g.B.rows = C1;
      g.M = C; g.N = Ca; g.K = Ci; g.batch = B;
      g.bn_hint = 128;
      g.D = s.Qb; g.ldd = Ca; g.strideD = CCa;
      GLF_TRY(gemm(g, stream));
    }
    GLF_TRY(gram_cvec(s.Wp, w->theta_b, s.cvec, B, C, Ci, stream));   // c_b = W'_b b_theta, kept in fp32
  }
  int np = 0;
  {  // U_b = X_b Q_b^T + c_b   (+ BatchNorm column statistics); bz stays folded into the BN affine
    GemmArgs g;
    g.A = opnd(X, 0, C, static_cast<long long>(N) * C);
    g.B = opnd(s.Qb, 0, Ca, CCa);
    g.M = N; g.N = C; g.K = C; g.batch = B;
    if (C % 256 == 0) g.bn_hint = 128;
    g.bias = s.cvec; g.bias_stride = C;
    g.D = s.U; g.ldd = C; g.strideD = static_cast<long long>(N) * C;
    g.colstats = (d->training && d->bn_layer) ? wf.colstats : nullptr;
    g.colstats_rows = &np;
    GLF_TRY(gemm(g, stream));
  }
  return bn_ln_fwd(d, m, X, w, np, z, s, wf, stream);
}

// Continues after the LayerNorm backward and bn_bwd_finalize: wb.dV, wb.k1..k3 are valid.
int tpavi_bwd_gram(const glf_desc* d, const Dims& m, const bf16* X, const glf_weights* w, const Saved& s, const WsBwd& wb,
                   void* dx, const glf_grads* g_, cudaStream_t stream) {
  const int C = m.C, Ci = m.Ci, Ca = m.Ca, C1 = m.C + 1;
  const int N = static_cast<int>(m.N), B = static_cast<int>(m.B);
  const long long CaCa = static_cast<long long>(Ca) * Ca, CiCa = static_cast<long long>(Ci) * Ca;
  const long long CCa = static_cast<long long>(C) * Ca, CiCi = static_cast<long long>(Ci) * Ci;
  const long long CCi = static_cast<long long>(C) * Ci, CC = static_cast<long long>(C) * C;
  const float invN = 1.f / static_cast<float>(N);
  const bool bn_train = d->bn_layer && d->training;   // k2, k3 != 0 only then
  // k1 * [R_b | rv_b]  with R_b = dV_b^T X_b, rv_b = dV_b^T 1: the BatchNorm-backward scale k1 (per channel of dV =
  // row of R) is applied in fp32 by the contraction's epilogue
  GLF_TRY(gram_token_contraction(wb.dV, X, wb.Rb, wb.Rf, wb.rv, s.sfv, wb.k1, static_cast<float>(N), B, N, C, Ca, wb.det,
                                 stream));
  // One CTA per sequence runs dQ~ -> dW' -> dM -> dT~ -> F (and E, e) in a single launch (glf_chain.cu); the four
  // weight-gradient sums over the sequences below then read its dQ~, dW', dM / N and dT~.
  const bool chain = gram_chain_supported(C, Ci);
  if (chain)
    GLF_TRY(gram_chain_bwd(s.Sa, s.Qb, s.waug, s.wz, wb.Rb, s.sfv, s.cvec, wb.rv, wb.k1, wb.k2, wb.k3, w->theta_b,
                           w->phi_b, w->g_b, bn_train ? 1 : 0, wb.dQa, wb.dWpb, wb.dM, wb.dT, wb.EF, wb.evec, wb.dcv,
                           wb.dtv, B, N, stream));
  if (chain)   // dW~theta, dWz, dW~g, dW~phi: one launch of K-concatenated products + a fixed-order reduction
    GLF_TRY(gram_wgrad(s.Wp, wb.dQa, wb.dWpb, s.Mb, wb.dM, s.T, wb.dT, s.Sa, wb.dcv, s.tv, wb.dtv, s.sfv, wb.wpart, g_, B, N,
                       stream));
  // Qk = k2 Q~ (column C: k2 c + k3), E = k1 Q
  if (!chain) GLF_TRY(gram_kprep(s.Qb, s.cvec, wb.k1, wb.k2, wb.k3, wb.AK, wb.EF, B, C, Ca, stream));
  if (!chain) {  // dQ~_b = dU_b^T X~_b = Qk_b S~_b + k1 [R_b | rv_b]     [C x Ca]   (S~ is symmetric; the second term is the addend)
    GemmArgs g;
    g.A = opnd(wb.AK, 0, Ca, CCa);
    g.B = opnd(s.Sa, 0, Ca, CaCa);
    g.B.rows = C1;
    g.M = C; g.N = Ca; g.K = C1; g.batch = B;
    g.bn_hint = 128;
    g.addend = wb.Rb; g.ld_add = Ca; g.stride_add = CaCa;
    g.D = wb.dQa; g.ldd = Ca; g.strideD = CCa;
    GLF_TRY(gemm(g, stream));
  }
  if (!chain) {  // dW'_b = dQ~_b W~theta^T               [C x Ci]
    GemmArgs g;
    g.A = opnd(wb.dQa, 0, Ca, CCa);
    g.B = opnd(s.waug, 0, Ca, 0);
    g.M = C; g.N = Ci; g.K = C1; g.batch = B;
    g.D = wb.dWpb; g.ldd = Ci; g.strideD = CCi;
    GLF_TRY(gemm(g, stream));
  }
  if (!chain) GLF_TRY(check_cuda(cudaMemsetAsync(wb.dwaug, 0, sizeof(float) * 3 * CiCa, stream), "memset dW~"));
  if (!chain) {  // dW~theta = sum_b W'_b^T dQ~_b         [Ci x Ca]   (batch reduced by fp32 red.add)
    GemmArgs g;
    g.A = opnd(s.Wp, 1, Ci, CCi);
    g.B = opnd(wb.dQa, 1, Ca, CCa);
    g.B.rows = C1;
    g.M = Ci; g.N = Ca; g.K = C; g.batch = B;
    g.bn_hint = 128;
    g.out_kind = 2;
    g.det = wb.det;
    g.D = wb.dwaug; g.ldd = Ca; g.strideD = 0;
    GLF_TRY(gemm(g, stream));
  }
  if (!chain) GLF_TRY(check_cuda(cudaMemsetAsync(g_->wz_w, 0, sizeof(float) * CCi, stream), "memset dWz"));
  if (!chain) {  // dWz = sum_b dW'_b M_b
    GemmArgs g;
    g.A = opnd(wb.dWpb, 0, Ci, CCi);
    g.B = opnd(s.Mb, 1, Ci, CiCi);
    g.M = C; g.N = Ci; g.K = Ci; g.batch = B;
    g.out_kind = 2;
    g.det = wb.det;
    g.D = g_->wz_w; g.ldd = Ci; g.strideD = 0;
    GLF_TRY(gemm(g, stream));
  }
  if (!chain) {  // dM_b = dW'_b^T Wz                     [Ci x Ci]
    GemmArgs g;
    g.A = opnd(wb.dWpb, 1, Ci, CCi);
    g.B = opnd(s.wz, 1, Ci, 0);
    g.M = Ci; g.N = Ci; g.K = C; g.batch = B;
    g.D = wb.dM; g.ldd = Ci; g.strideD = CiCi;
    GLF_TRY(gemm(g, stream));
  }
  if (!chain) {  // dW~g = sum_b (dM_b / N)^T T_b         [Ci x Ca]
    GemmArgs g;
    g.A = opnd(wb.dM, 1, Ci, CiCi);
    g.B = opnd(s.T, 1, Ca, CiCa);
    g.B.rows = C1;
    g.M = Ci; g.N = Ca; g.K = Ci; g.batch = B;
    g.bn_hint = 128;
    g.alpha = invN;
    g.out_kind = 2;
    g.det = wb.det;
    g.D = wb.dwaug + 2 * CiCa; g.ldd = Ca; g.strideD = 0;
    GLF_TRY(gemm(g, stream));
  }
  if (!chain) {  // dT_b = (dM_b / N) W~g                 [Ci x Ca]
    GemmArgs g;
    g.A = opnd(wb.dM, 0, Ci, CiCi);
    g.B = opnd(s.waug + 2 * CiCa, 1, Ca, 0);
    g.B.rows = C1;
    g.M = Ci; g.N = Ca; g.K = Ci; g.batch = B;
    g.bn_hint = 128;
    g.alpha = invN;
    g.D = wb.dT; g.ldd = Ca; g.strideD = CiCa;
    GLF_TRY(gemm(g, stream));
  }
  if (!chain) {  // dW~phi = sum_b dT_b S~_b              [Ci x Ca]
    GemmArgs g;
    g.A = opnd(wb.dT, 0, Ca, CiCa);
    g.B = opnd(s.Sa, 0, Ca, CaCa);
    g.B.rows = C1;
    g.M = Ci; g.N = Ca; g.K = C1; g.batch = B;
    g.bn_hint = 128;
    g.out_kind = 2;
    g.det = wb.det;
    g.D = wb.dwaug + CiCa; g.ldd = Ca; g.strideD = 0;
    GLF_TRY(gemm(g, stream));
  }
  if (!chain) {  // G0_b = dS~_b[:C, :] = W_phi^T dT_b     [C x Ca]   (row C is only needed for e: formed in gram_assemble_F)
    GemmArgs g;
    g.A = opnd(s.waug + CiCa, 1, Ca, 0);
    g.B = opnd(wb.dT, 1, Ca, CiCa);
    g.B.rows = C1;
    g.M = C; g.N = Ca; g.K = Ci; g.batch = B;
    g.bn_hint = 128;
    g.D = wb.G0; g.ldd = Ca; g.strideD = CCa;
    GLF_TRY(gemm(g, stream));
  }
  if (bn_train && !chain) {  // H_b = Q_b^T Qk_b    [C x Ca]  (dU Q = dV E + X H[:C,:C] + 1 H[:C,C]^T: the k2 U + k3 part of dU)
    GemmArgs g;
    g.A = opnd(s.Qb, 1, Ca, CCa);
    g.B = opnd(wb.AK, 1, Ca, CCa);
    g.B.rows = C1;
    g.M = C; g.N = Ca; g.K = C; g.batch = B;
    g.bn_hint = 128;
    g.D = wb.Hf; g.ldd = Ca; g.strideD = CCa;
    GLF_TRY(gemm(g, stream));
  }
  // F = (G0 + G0^T + H)[:C, :C] ;  e = (G0[:, C] + G0[C, :] + H[:, C])[:C]
  if (!chain) GLF_TRY(gram_assemble_F(wb.G0, bn_train ? wb.Hf : nullptr, wb.dT, s.waug + CiCa, wb.EF, wb.evec, B, C, Ci, Ca, stream));
  {  // dX_b = dV_b E_b + X_b F_b + 1 e_b^T + dV_b
    GemmArgs g;
    g.A = opnd(nullptr, 0, C, static_cast<long long>(N) * C);
    g.B = opnd(nullptr, 1, C, 2 * CC);
    g.M = N; g.N = C; g.K = C; g.batch = B;
    if (C % 256 == 0) g.bn_hint = 128;
    g.bias = wb.evec; g.bias_stride = C;
    // (the chain folds the residual dV into its E' = E + I)
    if (!chain) { g.addend = wb.dV; g.ld_add = C; g.stride_add = static_cast<long long>(N) * C; }
    g.D = m.pack_x ? static_cast<void*>(wb.dxtok) : dx; g.ldd = C; g.strideD = static_cast<long long>(N) * C;
    GLF_TRY(gemm_pair2(g, wb.dV, X, wb.EF, wb.EF + CC, stream));
  }
  if (!chain) GLF_TRY(gram_unpack_grads(wb.dwaug, g_, C, Ci, Ca, stream));
  if (m.pack_x)
    GLF_TRY(unpack_tokens(m, wb.dxtok, GLF_DTYPE_BF16, dx, d->x_layout == GLF_LAYOUT_NCTHW, d->io_dtype, stream));
  return 0;
}

// Bias gradients out[i] = column sums (the first n columns) of table i of `cs`: one fixed-order pass when the tables are
// short (one row per CTA) and of one length, else a stage-1 reduction first
int reduce_bias_grads(const ColTables& cs, int n, float* red1, float* const* out, cudaStream_t stream) {
  int np = cs.rows[0];
  long long rs = cs.stride;
  bool one_pass = np <= 4 * REDUCE_STAGE1_ROWS;
  for (int i = 1; i < cs.n; ++i) one_pass = one_pass && cs.rows[i] == np;
  const float *t0 = cs.tab[0], *t1 = cs.tab[1], *t2 = cs.tab[2];
  if (!one_pass) {
    GLF_TRY(reduce_stage1(t0, t1, t2, cs.n, cs.rows, &np, &rs, 0, 1, n, red1, stream));
    const long long pitch = static_cast<long long>(REDUCE_STAGE1_ROWS) * n;
    t0 = red1; t1 = red1 + pitch; t2 = red1 + 2 * pitch;
  }
  if (cs.n == 1) return reduce_partials(t0, np, rs, n, 1.f, out[0], stream);
  return reduce_partials3(t0, t1, t2, np, rs, n, out[0], out[1], out[2], stream);
}

// Scratch of the standalone attention entry points: the same pieces, sized the same way, as ws_bwd / ws_fwd give the
// module's attention (attention scratch, delta, the three column-statistic tables and the reduction buffer).
// C > 0 (mode='gaussian'): also the [B * N, 2C] pair dS X | dS^T X that the backward sums into dX.
struct WsAttn { void* attn; float *delta, *cs_t, *cs_p, *cs_g, *red1; bf16* dx2; int cs_cap_rows; };
size_t carve_ws_attn(long long B, long long N, int Ci, bool backward, void* base, WsAttn* w, int C = 0) {
  Carver c(base);
  w->attn = c.take<uint8_t>(attn_scratch_bytes(B, N, backward));
  w->delta = w->cs_t = w->cs_p = w->cs_g = w->red1 = nullptr;
  w->dx2 = (backward && C > 0) ? c.take<bf16>(static_cast<size_t>(B * N) * 2 * C) : nullptr;
  w->cs_cap_rows = 4 * static_cast<int>(B) * gemm_tiles_m(static_cast<int>(N));   // one partial per (tile, 32-row quarter)
  if (backward) {
    const size_t np = static_cast<size_t>(w->cs_cap_rows);
    w->delta = c.take<float>(static_cast<size_t>(B * N));
    w->cs_t = c.take<float>(np * 2 * Ci);
    w->cs_p = c.take<float>(np * 2 * Ci);
    w->cs_g = c.take<float>(np * 2 * Ci);
    w->red1 = c.take<float>(static_cast<size_t>(REDUCE_STAGE1_ROWS) * 3 * Ci);
  }
  return (c.off + 255) & ~static_cast<size_t>(255);
}

// the limits make_dims puts on a TPAVIModule's attention
int check_attn_dims(int B, int N, int Ci) {
  if (B <= 0 || N <= 0) return set_error(GLF_ERR_INVALID, "attention: empty input (B and N must be > 0, got %d, %d)", B, N);
  if (Ci <= 0 || Ci % 8 != 0 || Ci > 2048)
    return set_error(GLF_ERR_INVALID, "attention: Ci must be a positive multiple of 8, at most 2048 (got %d)", Ci);
  if (static_cast<long long>(B) * N > 0x7fffff00LL || 4LL * B * gemm_tiles_m(N) > 0x7fffffffLL)
    return set_error(GLF_ERR_INVALID, "attention: too many tokens");
  return 0;
}

int check_scratch(const void* scratch) {
  GLF_TRY(check_ptr(scratch, "scratch"));
  if ((reinterpret_cast<uintptr_t>(scratch) & 255) != 0) return set_error(GLF_ERR_WORKSPACE, "scratch must be 256-byte aligned");
  return 0;
}

}  // namespace
}  // namespace glf

using namespace glf;

extern "C" {

GLF_API int glf_version(void) { return GLF_VERSION; }
GLF_API const char* glf_last_error(void) { return g_err; }

GLF_API int glf_tpavi_sizes(const glf_desc* d, glf_sizes* out) {
  Dims m;
  GLF_TRY(make_dims(d, &m));
  if (out == nullptr) return set_error(GLF_ERR_INVALID, "out is NULL");
  if (d->precision == GLF_PRECISION_F32X3) return tpavi_sizes_f32x3(d, m, out);
  Saved s; WsFwd wf; WsBwd wb;
  out->saved_bytes = carve_saved(m, nullptr, &s);
  out->ws_fwd_bytes = carve_ws_fwd(m, nullptr, &wf, out->saved_bytes);
  out->ws_bwd_bytes = carve_ws_bwd(d, m, nullptr, &wb);
  return 0;
}

GLF_API int glf_tpavi_fwd(const glf_desc* d, const void* x, const glf_weights* w, void* z, void* saved, void* ws,
                  glf_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  Dims m;
  GLF_TRY(make_dims(d, &m));
  GLF_TRY(check_device_sm100());
  GLF_TRY(check_ptr(x, "x"));
  GLF_TRY(check_ptr(z, "z"));
  GLF_TRY(check_ptr(ws, "ws"));
  if (w == nullptr) return set_error(GLF_ERR_INVALID, "weights is NULL");
  if ((reinterpret_cast<uintptr_t>(ws) & 255) != 0 || (saved && (reinterpret_cast<uintptr_t>(saved) & 255) != 0))
    return set_error(GLF_ERR_WORKSPACE, "saved/ws blobs must be 256-byte aligned");
  if (d->precision == GLF_PRECISION_F32X3) return tpavi_fwd_f32x3(d, m, x, w, z, saved, ws, stream);
  Saved s; WsFwd wf;
  const size_t saved_bytes = carve_saved(m, nullptr, &s);
  carve_ws_fwd(m, ws, &wf, saved_bytes);
  carve_saved(m, saved ? saved : wf.saved_fallback, &s);
  if (m.half_params) GLF_TRY(stage_params(m, w, s.pshadow, stream));
  const glf_weights w32 = fp32_weights(m, w, s.pshadow);
  w = &w32;
  if (m.gram) return tpavi_fwd_gram(d, m, x, w, z, s, wf, stream);
  const int C = m.C, Ci = m.Ci;
  const int N = static_cast<int>(m.N), rows = static_cast<int>(m.rows), B = static_cast<int>(m.B);

  if (m.gauss)
    GLF_TRY(prep_weights_gaussian(w, C, Ci, s.wcat, s.wcatT, s.bcat, s.wz, s.wzT, stream));
  else
    GLF_TRY(prep_weights(w, C, Ci, s.wcat, s.wcatT, s.bcat, s.wz, s.wzT, stream));
  const bf16* X = reinterpret_cast<const bf16*>(x);
  if (m.pack_x) {
    GLF_TRY(pack_tokens(m, x, d->io_dtype, d->x_layout == GLF_LAYOUT_NCTHW, s.xtok, GLF_DTYPE_BF16, stream));
    X = s.xtok;
  }
  const int Pw = m.gauss ? Ci : 3 * Ci;
  {  // P = X Wcat^T + bcat   (gaussian: G = X Wg^T + bg)
    GemmArgs g;
    g.A = opnd(X, 0, C, 0);
    g.B = opnd(s.wcat, 0, C, 0);
    g.M = rows; g.N = Pw; g.K = C;
    g.bias = s.bcat;
    g.D = s.P; g.ldd = Pw;
    GLF_TRY(gemm(g, stream));
  }
  int np = 0;
  if (m.dot) {
    const long long CiCi = static_cast<long long>(Ci) * Ci;
    {  // M_b[i,j] = sum_n Phi[n,i] G[n,j] / N      (token contraction: both operands MN-major views of P)
      GemmArgs g;
      g.A = opnd(s.P + Ci, 1, 3 * Ci, static_cast<long long>(N) * 3 * Ci);
      g.B = opnd(s.P + 2 * Ci, 1, 3 * Ci, static_cast<long long>(N) * 3 * Ci);
      g.M = Ci; g.N = Ci; g.K = N; g.batch = B;
      g.alpha = 1.f / static_cast<float>(N);
      g.det = wf.det;
      GLF_TRY(token_contraction(g, s.Mb, wf.Mf, stream));
    }
    {  // W'_b[c,i] = sum_j Wz[c,j] M_b[i,j]        (folds Y = Theta M and U = Y Wz^T into one product per token)
      GemmArgs g;
      g.A = opnd(s.wz, 0, Ci, 0);
      g.B = opnd(s.Mb, 0, Ci, CiCi);
      g.M = C; g.N = Ci; g.K = Ci; g.batch = B;
      g.D = s.Wp; g.ldd = Ci; g.strideD = static_cast<long long>(C) * Ci;
      GLF_TRY(gemm(g, stream));
    }
    {  // U_b = Theta_b W'_b^T   (+ BatchNorm column statistics); the bias bz is folded into the BN affine (bn_finalize)
      GemmArgs g;
      g.A = opnd(s.P, 0, 3 * Ci, static_cast<long long>(N) * 3 * Ci);
      g.B = opnd(s.Wp, 0, Ci, static_cast<long long>(C) * Ci);
      g.M = N; g.N = C; g.K = Ci; g.batch = B;
      g.D = s.U; g.ldd = C; g.strideD = static_cast<long long>(N) * C;
      g.colstats = (d->training && d->bn_layer) ? wf.colstats : nullptr;
      g.colstats_rows = &np;
      GLF_TRY(gemm(g, stream));
    }
  } else {
    if (m.gauss)   // Y = softmax(X X^T) G
      GLF_TRY(attn_fwd(attn_args_gaussian(X, s.P, nullptr, nullptr, nullptr, 0, 0, C, Ci), s.Y, s.lse, B, N, wf.attn,
                       stream));
    else
      GLF_TRY(flash_fwd(s.P, s.Y, s.lse, B, N, Ci, wf.attn, stream));
    {  // U = Y Wz^T   (bz folded into the BN affine)
      GemmArgs g;
      g.A = opnd(s.Y, 0, Ci, 0);
      g.B = opnd(s.wz, 0, Ci, 0);
      g.M = rows; g.N = C; g.K = Ci;
      g.D = s.U; g.ldd = C;
      g.colstats = (d->training && d->bn_layer) ? wf.colstats : nullptr;
      g.colstats_rows = &np;
      GLF_TRY(gemm(g, stream));
    }
  }
  return bn_ln_fwd(d, m, X, w, np, z, s, wf, stream);
}

GLF_API int glf_tpavi_bwd(const glf_desc* d, const void* dz, const void* x, const glf_weights* w, const void* saved, void* dx,
                  const glf_grads* g_, void* ws, glf_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  Dims m;
  GLF_TRY(make_dims(d, &m));
  GLF_TRY(check_device_sm100());
  GLF_TRY(check_ptr(dz, "dz"));
  GLF_TRY(check_ptr(x, "x"));
  GLF_TRY(check_ptr(dx, "dx"));
  GLF_TRY(check_ptr(saved, "saved"));
  GLF_TRY(check_ptr(ws, "ws"));
  if (w == nullptr || g_ == nullptr) return set_error(GLF_ERR_INVALID, "weights/grads is NULL");
  if ((reinterpret_cast<uintptr_t>(ws) & 255) != 0 || (reinterpret_cast<uintptr_t>(saved) & 255) != 0)
    return set_error(GLF_ERR_WORKSPACE, "saved/ws blobs must be 256-byte aligned");
  if (d->precision == GLF_PRECISION_F32X3) return tpavi_bwd_f32x3(d, m, dz, x, w, saved, dx, g_, ws, stream);
  Saved s; WsBwd wb;
  carve_saved(m, const_cast<void*>(saved), &s);
  carve_ws_bwd(d, m, ws, &wb);
  const glf_grads* g_out = g_;
  const glf_weights w32 = fp32_weights(m, w, s.pshadow);
  const glf_grads g32 = fp32_grads(m, g_, wb.gstage);
  w = &w32;
  g_ = &g32;
  const int C = m.C, Ci = m.Ci;
  const int N = static_cast<int>(m.N), rows = static_cast<int>(m.rows), B = static_cast<int>(m.B);
  const bf16* X = m.pack_x ? s.xtok : reinterpret_cast<const bf16*>(x);
  const long long seqP = static_cast<long long>(N) * 3 * Ci;

  const void* dZ = dz;
  int dz_dtype = d->io_dtype;
  if (m.pack_dz && !defer_ln(d)) {
    GLF_TRY(pack_tokens(m, dz, d->io_dtype, /*ncthw=*/true, wb.dztok, GLF_DTYPE_BF16, stream));
    dZ = wb.dztok;
    dz_dtype = GLF_DTYPE_BF16;
  }
  int nb = 0;
  if (defer_ln(d)) {
    // dV and the partials were written by glf_fusion_ln_bwd
    nb = ln_tma_supported(C) ? ln_bwd_tma_blocks(m.rows) : bn_res_ln_bwd_blocks(m.rows, C);
  } else {
    GLF_TRY(bn_res_ln_bwd(dZ, dz_dtype, s.U, X, GLF_DTYPE_BF16, s.bn_a, s.bn_b, s.bn_mean, s.bn_rstd, w->ln_w, s.ln_mu,
                          s.ln_r, wb.dV, wb.part_ln, m.rows, C, &nb, stream));
  }
  GLF_TRY(bn_bwd_finalize(wb.part_ln, nb, C, static_cast<double>(m.rows), d, w, s.bn_mean, s.bn_rstd, g_, wb.k1, wb.k2,
                          wb.k3, stream));
  if (m.gram) {
    GLF_TRY(tpavi_bwd_gram(d, m, X, w, s, wb, dx, g_, stream));
    return emit_grads(m, wb.gstage, g_out, stream);
  }
  const bf16* dU = wb.dV;
  if (d->bn_layer) {
    GLF_TRY(bn_bwd_apply(wb.dV, s.U, GLF_DTYPE_BF16, wb.k1, wb.k2, wb.k3, wb.dU, m.rows, C, stream));
    dU = wb.dU;
  }
  ColTables cs;
  if (m.dot) {   // three GEMM epilogues: their row counts can differ (tile shape and grid differ per product)
    cs.n = 3;
    cs.tab[0] = wb.cs_t; cs.tab[1] = wb.cs_p; cs.tab[2] = wb.cs_g;
    cs.stride = 2LL * Ci;
    const long long CiCi = static_cast<long long>(Ci) * Ci;
    const long long CCi = static_cast<long long>(C) * Ci;
    {  // dTheta_b = dU_b W'_b          (B operand = W'_b read MN-major: stored [K=c][N=i])
      GemmArgs g;
      g.A = opnd(dU, 0, C, static_cast<long long>(N) * C);
      g.B = opnd(s.Wp, 1, Ci, CCi);
      g.M = N; g.N = Ci; g.K = C; g.batch = B;
      g.D = wb.dP; g.ldd = 3 * Ci; g.strideD = seqP;
      g.colstats = wb.cs_t;
      g.colstats_rows = &cs.rows[0];
      GLF_TRY(gemm(g, stream));
    }
    {  // dW'_b[c,i] = sum_n dU[n,c] Theta[n,i]
      GemmArgs g;
      g.A = opnd(dU, 1, C, static_cast<long long>(N) * C);
      g.B = opnd(s.P, 1, 3 * Ci, seqP);
      g.M = C; g.N = Ci; g.K = N; g.batch = B;
      g.det = wb.det;
      GLF_TRY(token_contraction(g, wb.dWpb, wb.dWpf, stream));
    }
    GLF_TRY(check_cuda(cudaMemsetAsync(g_->wz_w, 0, sizeof(float) * CCi, stream), "memset dWz"));
    {  // dWz[c,j] = sum_b sum_i dW'_b[c,i] M_b[i,j]     (batch reduced by fp32 red.add into one output)
      GemmArgs g;
      g.A = opnd(wb.dWpb, 0, Ci, CCi);
      g.B = opnd(s.Mb, 1, Ci, CiCi);
      g.M = C; g.N = Ci; g.K = Ci; g.batch = B;
      g.out_kind = 2;
      g.det = wb.det;
      g.D = g_->wz_w; g.ldd = Ci; g.strideD = 0;
      GLF_TRY(gemm(g, stream));
    }
    {  // dM_b[i,j] = sum_c dW'_b[c,i] Wz[c,j]
      GemmArgs g;
      g.A = opnd(wb.dWpb, 1, Ci, CCi);
      g.B = opnd(s.wz, 1, Ci, 0);
      g.M = Ci; g.N = Ci; g.K = C; g.batch = B;
      g.D = wb.dM; g.ldd = Ci; g.strideD = CiCi;
      GLF_TRY(gemm(g, stream));
    }
    {  // dPhi_b = G_b dM_b^T / N
      GemmArgs g;
      g.A = opnd(s.P + 2 * Ci, 0, 3 * Ci, seqP);
      g.B = opnd(wb.dM, 0, Ci, CiCi);
      g.M = N; g.N = Ci; g.K = Ci; g.batch = B;
      g.alpha = 1.f / static_cast<float>(N);
      g.D = wb.dP + Ci; g.ldd = 3 * Ci; g.strideD = seqP;
      g.colstats = wb.cs_p;
      g.colstats_rows = &cs.rows[1];
      GLF_TRY(gemm(g, stream));
    }
    {  // dG_b = Phi_b dM_b / N          (B operand = dM_b read MN-major)
      GemmArgs g;
      g.A = opnd(s.P + Ci, 0, 3 * Ci, seqP);
      g.B = opnd(wb.dM, 1, Ci, CiCi);
      g.M = N; g.N = Ci; g.K = Ci; g.batch = B;
      g.alpha = 1.f / static_cast<float>(N);
      g.D = wb.dP + 2 * Ci; g.ldd = 3 * Ci; g.strideD = seqP;
      g.colstats = wb.cs_g;
      g.colstats_rows = &cs.rows[2];
      GLF_TRY(gemm(g, stream));
    }
  } else {
    {  // dY = dU Wz
      GemmArgs g;
      g.A = opnd(dU, 0, C, 0);
      g.B = opnd(s.wzT, 0, C, 0);
      g.M = rows; g.N = Ci; g.K = C;
      g.D = wb.dY; g.ldd = Ci;
      GLF_TRY(gemm(g, stream));
    }
    GLF_TRY(check_cuda(cudaMemsetAsync(g_->wz_w, 0, sizeof(float) * C * Ci, stream), "memset dWz"));
    {  // dWz[c,j] = sum_n dU[n,c] Y[n,j]
      GemmArgs g;
      g.A = opnd(dU, 1, C, 0);
      g.B = opnd(s.Y, 1, Ci, 0);
      g.M = C; g.N = Ci; g.K = rows;
      g.out_kind = 2;
      g.det = wb.det;
      g.D = g_->wz_w; g.ldd = Ci;
      g.split_k = pick_split_rounds(C, Ci, 1, rows);
      GLF_TRY(gemm(g, stream));
    }
    if (m.gauss) {   // dP = [dS X | dS^T X | dG]: the two attention terms of dX side by side, summed by the dX product
      const long long ldp = 2LL * C + Ci;
      const AttnArgs a = attn_args_gaussian(X, s.P, wb.dP, wb.dP + C, wb.dP + 2 * C, ldp, ldp, C, Ci);
      GLF_TRY(attn_bwd(a, s.Y, wb.dY, s.lse, wb.delta, wb.cs_t, wb.cs_p, wb.cs_g, 4 * B * m.tiles_seq, &cs, B, N,
                       wb.attn, stream));
    } else {
      GLF_TRY(flash_bwd(s.P, s.Y, wb.dY, s.lse, wb.dP, wb.delta, wb.cs_t, wb.cs_p, wb.cs_g, 4 * B * m.tiles_seq, &cs,
                        B, N, Ci, wb.attn, stream));
    }
  }
  // dP columns [wrow, ldp) are the projection gradients (all three, or dG alone for gaussian)
  const int ldp = m.gauss ? 2 * C + Ci : 3 * Ci;
  const int wrow = m.gauss ? 2 * C : 0;
  const int nproj = m.gauss ? Ci : 3 * Ci;
  GLF_TRY(check_cuda(cudaMemsetAsync(wb.dwcat, 0, sizeof(float) * nproj * C, stream), "memset dWcat"));
  {  // dWcat[r,c] = sum_n dP[n,r] X[n,c]
    GemmArgs g;
    g.A = opnd(wb.dP + wrow, 1, ldp, 0);
    g.B = opnd(X, 1, C, 0);
    g.M = nproj; g.N = C; g.K = rows;
    g.out_kind = 2;
    g.det = wb.det;
    g.D = wb.dwcat; g.ldd = C;
    g.split_k = pick_split_rounds(nproj, C, 1, rows);
    GLF_TRY(gemm(g, stream));
  }
  GLF_TRY(scatter_proj_grads(wb.dwcat, g_, C, Ci, m.gauss, stream));
  {  // dX = dP Wcat + dV   (gaussian: [dS X | dS^T X | dG] [I | I | Wg^T]^T + dV, each attention term rounded to bf16
     // once before this fp32 sum)
    GemmArgs g;
    g.A = opnd(wb.dP, 0, ldp, 0);
    g.B = opnd(s.wcatT, 0, ldp, 0);
    g.M = rows; g.N = C; g.K = ldp;
    g.addend = wb.dV; g.ld_add = C;
    g.D = m.pack_x ? static_cast<void*>(wb.dxtok) : dx; g.ldd = C;
    GLF_TRY(gemm(g, stream));
  }
  float* const db[3] = {g_->theta_b, g_->phi_b, g_->g_b};
  GLF_TRY(reduce_bias_grads(cs, Ci, wb.red1, m.gauss ? db + 2 : db, stream));   // gaussian: the g bias alone
  if (m.pack_x)
    GLF_TRY(unpack_tokens(m, wb.dxtok, GLF_DTYPE_BF16, dx, d->x_layout == GLF_LAYOUT_NCTHW, d->io_dtype, stream));
  return emit_grads(m, wb.gstage, g_out, stream);
}

GLF_API int glf_fusion_ln_supported(const glf_desc* d) {
  Dims m;
  if (make_dims(d, &m) != 0) return 0;
  return check_pair(d, m) == 0 ? 1 : 0;
}

GLF_API int glf_fusion_ln_fwd(const glf_desc* d, const void* xg, const void* xl, const glf_weights* wg,
                              const glf_weights* wl, void* z, void* saved_g, void* saved_l, glf_stream_t stream_) {
  return glf_fusion_ln_fwd_parts(d, xg, xl, wg, wl, z, nullptr, saved_g, saved_l, stream_);
}

GLF_API int glf_fusion_ln_fwd_parts(const glf_desc* d, const void* xg, const void* xl, const glf_weights* wg,
                                    const glf_weights* wl, void* z, void* z_global, void* saved_g, void* saved_l,
                                    glf_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if (z_global != nullptr) {
    GLF_TRY(check_ptr(z_global, "z_global"));
    if (d != nullptr && d->accumulate) return set_error(GLF_ERR_INVALID, "glf_fusion_ln_fwd_parts: accumulate is not supported");
  }
  Dims m;
  GLF_TRY(make_dims(d, &m));
  GLF_TRY(check_device_sm100());
  GLF_TRY(check_pair(d, m));
  GLF_TRY(check_ptr(xg, "xg"));
  GLF_TRY(check_ptr(xl, "xl"));
  GLF_TRY(check_ptr(z, "z"));
  GLF_TRY(check_ptr(saved_g, "saved_g"));
  GLF_TRY(check_ptr(saved_l, "saved_l"));
  if (wg == nullptr || wl == nullptr) return set_error(GLF_ERR_INVALID, "weights is NULL");
  const LnPair p = ln_pair(m, xg, xl, wg, wl, saved_g, saved_l);
  if (!ln_tma_supported(m.C))     // wide rows (256 < C <= 2048): the sliced-row ring kernel, both blocks in one pass
    return ln_pair_fwd_wide(p.U, p.X, p.a, p.b, p.lw, p.lb, p.mu, p.r, z, m.rows, m.C, d->eps_ln, d->accumulate, stream,
                            z_global, pair_z_dtype(d));
  return ln_fwd_tma(2, p.U, p.X, p.a, p.b, p.lw, p.lb, p.mu, p.r, z, m.rows, m.C, d->eps_ln, d->accumulate, stream,
                    z_global, pair_z_dtype(d));
}

GLF_API int glf_fusion_ln_bwd(const glf_desc* d, const void* dz, const void* xg, const void* xl, const glf_weights* wg,
                              const glf_weights* wl, const void* saved_g, const void* saved_l, void* ws_g, void* ws_l,
                              glf_stream_t stream_) {
  return glf_fusion_ln_bwd_views(d, dz, nullptr, nullptr, xg, xl, wg, wl, saved_g, saved_l, ws_g, ws_l, stream_);
}

GLF_API int glf_fusion_ln_bwd_views_supported(const glf_desc* d) {
  Dims m;
  if (d == nullptr || make_dims(d, &m) != 0 || check_pair(d, m) != 0 || !ln_tma_supported(m.C)) return 0;
  return (static_cast<long long>(d->H) * d->W) % ln_bwd_tma_tile_rows() == 0 && d->T <= 8 ? 1 : 0;
}

GLF_API int glf_fusion_ln_bwd_views(const glf_desc* d, const void* dz, const void* const* dz_views,
                                    const int64_t* dz_stride_b, const void* xg, const void* xl, const glf_weights* wg,
                                    const glf_weights* wl, const void* saved_g, const void* saved_l, void* ws_g,
                                    void* ws_l, glf_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  Dims m;
  GLF_TRY(make_dims(d, &m));
  GLF_TRY(check_device_sm100());
  GLF_TRY(check_pair(d, m));
  const bool views = dz_views != nullptr;
  if (views && dz_stride_b == nullptr) return set_error(GLF_ERR_INVALID, "dz_stride_b is NULL");
  if (!views) GLF_TRY(check_ptr(dz, "dz"));
  GLF_TRY(check_ptr(xg, "xg"));
  GLF_TRY(check_ptr(xl, "xl"));
  GLF_TRY(check_ptr(saved_g, "saved_g"));
  GLF_TRY(check_ptr(saved_l, "saved_l"));
  GLF_TRY(check_ptr(ws_g, "ws_g"));
  GLF_TRY(check_ptr(ws_l, "ws_l"));
  if (wg == nullptr || wl == nullptr) return set_error(GLF_ERR_INVALID, "weights is NULL");
  const LnPair p = ln_pair(m, xg, xl, wg, wl, saved_g, saved_l);
  WsBwd bg, bl;
  carve_ws_bwd(d, m, ws_g, &bg);
  carve_ws_bwd(d, m, ws_l, &bl);
  bf16* dV[2] = {bg.dV, bl.dV};
  float* part[2] = {bg.part_ln, bl.part_ln};
  int nb = 0;
  static_assert(sizeof(long long) == sizeof(int64_t), "stride tables are passed through unchanged");
  if (!ln_tma_supported(m.C)) {
    // wide rows: the backward is issue-bound, not bandwidth-bound (DESIGN.md), so sharing the dz read buys nothing;
    // the two blocks run the sliced-row ring kernel one after the other
    if (views) return set_error(GLF_ERR_UNSUPPORTED, "per-view dz needs C <= 256");
    for (int k = 0; k < 2; ++k)
      GLF_TRY(bn_res_ln_bwd(dz, pair_z_dtype(d), p.U[k], p.X[k], GLF_DTYPE_BF16, p.a[k], p.b[k], p.mean[k], p.rstd[k],
                            p.lw[k], p.mu[k], p.r[k], dV[k], part[k], m.rows, m.C, &nb, stream));
    return 0;
  }
  return ln_bwd_tma(2, dz, p.U, p.X, p.a, p.b, p.lw, p.mean, p.rstd, p.mu, p.r, dV, part, m.rows, m.C, &nb, stream,
                    views ? d->T : 0, dz_views, reinterpret_cast<const long long*>(dz_stride_b), d->H * d->W, pair_z_dtype(d));
}

GLF_API int glf_gate_concat_fwd(int B, int C, int V, int h, int w, int ncls, float weight, int io_dtype, int x_dtype,
                        const void* const* f4, const float* const* cls, const float* const* ctr, void* xg, void* xl,
                        float* gate, glf_stream_t stream) {
  GLF_TRY(check_device_sm100());
  if (B <= 0 || C <= 0 || h <= 0 || w <= 0 || ncls <= 0) return set_error(GLF_ERR_INVALID, "gate_concat: empty input");
  if (f4 == nullptr || cls == nullptr || ctr == nullptr) return set_error(GLF_ERR_INVALID, "gate_concat: NULL pointer table");
  GLF_TRY(check_ptr(xg, "xg"));
  GLF_TRY(check_ptr(xl, "xl"));
  return gate_concat_fwd(B, C, V, h, w, ncls, weight, io_dtype, x_dtype, f4, cls, ctr, xg, xl, gate,
                         reinterpret_cast<cudaStream_t>(stream));
}

GLF_API int glf_gate_concat_bwd(int B, int C, int V, int h, int w, int ncls, float weight, int io_dtype, int x_dtype,
                        const void* const* f4, const float* const* cls, const float* const* ctr, const float* gate,
                        const void* dxg, const void* dxl, void* const* df4, float* const* dcls, float* const* dctr,
                        void* scratch, glf_stream_t stream) {
  GLF_TRY(check_device_sm100());
  if (B <= 0 || C <= 0 || h <= 0 || w <= 0 || ncls <= 0) return set_error(GLF_ERR_INVALID, "gate_concat: empty input");
  if (f4 == nullptr || cls == nullptr || ctr == nullptr || df4 == nullptr || dcls == nullptr || dctr == nullptr)
    return set_error(GLF_ERR_INVALID, "gate_concat: NULL pointer table");
  GLF_TRY(check_ptr(dxg, "dxg"));
  GLF_TRY(check_ptr(dxl, "dxl"));
  return gate_concat_bwd(B, C, V, h, w, ncls, weight, io_dtype, x_dtype, f4, cls, ctr, gate, dxg, dxl, df4, dcls, dctr,
                         reinterpret_cast<float*>(scratch), reinterpret_cast<cudaStream_t>(stream));
}

GLF_API size_t glf_gate_concat_bwd_scratch_bytes(int B, int C, int V, int h, int w) {
  return gate_bwd_scratch_bytes(B, C, V, h, w);
}

GLF_API int glf_gate_concat_cl_fwd(int B, int C, int V, int h, int w, int ncls, float weight, int io_dtype,
                                   const void* const* f4, const int64_t* stride_b, const int64_t* stride_t,
                                   const float* const* cls, const float* const* ctr, void* xg, void* xl, float* gate,
                                   glf_stream_t stream) {
  GLF_TRY(check_device_sm100());
  if (B <= 0 || C <= 0 || h <= 0 || w <= 0 || ncls <= 0) return set_error(GLF_ERR_INVALID, "gate_concat: empty input");
  if (f4 == nullptr || cls == nullptr || ctr == nullptr || stride_b == nullptr || stride_t == nullptr)
    return set_error(GLF_ERR_INVALID, "gate_concat: NULL table");
  GLF_TRY(check_ptr(xg, "xg"));
  GLF_TRY(check_ptr(xl, "xl"));
  return gate_concat_cl_fwd(B, C, V, h, w, ncls, weight, io_dtype, f4, reinterpret_cast<const long long*>(stride_b),
                            reinterpret_cast<const long long*>(stride_t), cls, ctr, xg, xl, gate,
                            reinterpret_cast<cudaStream_t>(stream));
}

GLF_API int glf_gate_concat_cl_bwd(int B, int C, int V, int h, int w, int ncls, float weight, int io_dtype,
                                   const void* const* f4, const int64_t* stride_b, const int64_t* stride_t,
                                   const float* const* cls, const float* const* ctr, const float* gate, const void* dxg,
                                   const void* dxl, void* const* df4, const int64_t* dstride_b, const int64_t* dstride_t,
                                   float* const* dcls, float* const* dctr, void* scratch, glf_stream_t stream) {
  GLF_TRY(check_device_sm100());
  if (B <= 0 || C <= 0 || h <= 0 || w <= 0 || ncls <= 0) return set_error(GLF_ERR_INVALID, "gate_concat: empty input");
  if (f4 == nullptr || cls == nullptr || ctr == nullptr || df4 == nullptr || dcls == nullptr || dctr == nullptr ||
      stride_b == nullptr || stride_t == nullptr || dstride_b == nullptr || dstride_t == nullptr)
    return set_error(GLF_ERR_INVALID, "gate_concat: NULL table");
  GLF_TRY(check_ptr(dxg, "dxg"));
  GLF_TRY(check_ptr(dxl, "dxl"));
  return gate_concat_cl_bwd(B, C, V, h, w, ncls, weight, io_dtype, f4, reinterpret_cast<const long long*>(stride_b),
                            reinterpret_cast<const long long*>(stride_t), cls, ctr, gate, dxg, dxl, df4,
                            reinterpret_cast<const long long*>(dstride_b), reinterpret_cast<const long long*>(dstride_t),
                            dcls, dctr, reinterpret_cast<float*>(scratch), reinterpret_cast<cudaStream_t>(stream));
}

GLF_API int glf_views_to_tokens(int B, int C, int V, int T, int src_dtype, const void* const* src,
                                const int64_t* stride_b, const int64_t* stride_c, const int64_t* stride_t, void* out,
                                glf_stream_t stream) {
  GLF_TRY(check_device_sm100());
  if (B <= 0 || C <= 0 || T <= 0) return set_error(GLF_ERR_INVALID, "views_to_tokens: empty input");
  if (src == nullptr || stride_b == nullptr || stride_c == nullptr || stride_t == nullptr)
    return set_error(GLF_ERR_INVALID, "views_to_tokens: NULL table");
  GLF_TRY(check_ptr(out, "out"));
  static_assert(sizeof(long long) == sizeof(int64_t), "stride tables are passed through unchanged");
  return views_to_tokens(B, C, V, T, src_dtype, src, reinterpret_cast<const long long*>(stride_b),
                         reinterpret_cast<const long long*>(stride_c), reinterpret_cast<const long long*>(stride_t), out,
                         reinterpret_cast<cudaStream_t>(stream));
}

GLF_API size_t glf_p2p_signal_bytes(int world) { return p2p_signal_bytes(world); }
GLF_API int64_t glf_p2p_max_floats(void) { return p2p_max_floats(); }
GLF_API int glf_p2p_export(const void* ptr, unsigned char handle[64], uint64_t* offset) {
  if (ptr == nullptr || handle == nullptr || offset == nullptr) return set_error(GLF_ERR_INVALID, "p2p_export: NULL argument");
  unsigned long long off = 0;
  GLF_TRY(p2p_export(ptr, handle, &off));
  *offset = off;
  return 0;
}
GLF_API int glf_p2p_open(const unsigned char handle[64], uint64_t offset, void** out) {
  if (handle == nullptr || out == nullptr) return set_error(GLF_ERR_INVALID, "p2p_open: NULL argument");
  return p2p_open(handle, offset, out);
}
GLF_API int glf_p2p_close(void* ptr, uint64_t offset) {
  if (ptr == nullptr) return set_error(GLF_ERR_INVALID, "p2p_close: NULL argument");
  return p2p_close(ptr, offset);
}
GLF_API int glf_p2p_allreduce(void* const* bufs, void* const* sigs, int rank, int world, int64_t n, float scale,
                      glf_stream_t stream) {
  GLF_TRY(check_device_sm100());
  if (bufs == nullptr || sigs == nullptr) return set_error(GLF_ERR_INVALID, "p2p_allreduce: NULL pointer table");
  return p2p_allreduce(bufs, sigs, rank, world, n, scale, reinterpret_cast<cudaStream_t>(stream));
}

GLF_API int glf_gemm_bf16(const void* A, const void* B, void* D, int M, int N, int K, int batch, int a_mn, int b_mn,
                  int64_t lda, int64_t ldb, int64_t ldd, int64_t strideA, int64_t strideB, int64_t strideD,
                  const float* bias, float alpha, const void* addend, int64_t ld_add, int64_t stride_add,
                  int out_kind, int split_k, float* colstats, glf_stream_t stream) {
  GLF_TRY(check_device_sm100());
  GLF_TRY(check_ptr(A, "A"));
  GLF_TRY(check_ptr(B, "B"));
  GLF_TRY(check_ptr(D, "D"));
  GemmArgs g;
  g.A = opnd(A, a_mn, lda, strideA);
  g.B = opnd(B, b_mn, ldb, strideB);
  g.M = M; g.N = N; g.K = K; g.batch = batch;
  g.alpha = alpha; g.bias = bias;
  g.out_kind = out_kind;
  g.D = D; g.ldd = ldd; g.strideD = strideD;
  g.addend = reinterpret_cast<const bf16*>(addend); g.ld_add = ld_add; g.stride_add = stride_add;
  g.colstats = colstats;
  g.split_k = split_k;
  return gemm(g, reinterpret_cast<cudaStream_t>(stream));
}

GLF_API int glf_gemm_bf16_ex(const void* A, const void* B, void* D, int M, int N, int K, int batch, int a_mn, int b_mn,
                     int64_t lda, int64_t ldb, int64_t ldd, int64_t strideA, int64_t strideB, int64_t strideD,
                     const float* bias, int64_t bias_stride, float alpha, int out_kind, int split_k, float* rowsum,
                     glf_stream_t stream) {
  GLF_TRY(check_device_sm100());
  GLF_TRY(check_ptr(A, "A"));
  GLF_TRY(check_ptr(B, "B"));
  GLF_TRY(check_ptr(D, "D"));
  GemmArgs g;
  g.A = opnd(A, a_mn, lda, strideA);
  g.B = opnd(B, b_mn, ldb, strideB);
  g.M = M; g.N = N; g.K = K; g.batch = batch;
  g.alpha = alpha; g.bias = bias; g.bias_stride = bias_stride;
  g.out_kind = out_kind;
  g.D = D; g.ldd = ldd; g.strideD = strideD;
  g.split_k = split_k;
  g.rowsum = rowsum; g.rowsum_stride = M;
  return gemm(g, reinterpret_cast<cudaStream_t>(stream));
}

GLF_API int glf_gram_contraction(const void* A, const void* X, void* D, float* colsum, int B, int N, int C, int ldd,
                         glf_stream_t stream) {
  GLF_TRY(check_device_sm100());
  GLF_TRY(check_ptr(A, "A"));
  GLF_TRY(check_ptr(X, "X"));
  GLF_TRY(check_ptr(D, "D"));
  GLF_TRY(check_ptr(colsum, "colsum"));
  if (B <= 0 || N <= 0) return set_error(GLF_ERR_INVALID, "gram_contraction: empty input");
  if (ldd < C || ldd % 8 != 0) return set_error(GLF_ERR_INVALID, "gram_contraction: ldd must be >= C and a multiple of 8");
  return gram_contraction(reinterpret_cast<const bf16*>(A), reinterpret_cast<const bf16*>(X), reinterpret_cast<bf16*>(D),
                          nullptr, colsum, nullptr, nullptr, 0.f, 0, B, N, C, ldd, 1,
                          reinterpret_cast<cudaStream_t>(stream));
}

GLF_API size_t glf_attention_scratch_bytes(int B, int N, int Ci, int backward) {
  if (check_attn_dims(B, N, Ci) != 0) return 0;
  WsAttn w;
  return carve_ws_attn(B, N, Ci, backward != 0, nullptr, &w);
}

GLF_API int glf_attention_fwd(const void* P3, void* Y, float* lse, int B, int N, int Ci, void* scratch,
                              glf_stream_t stream) {
  GLF_TRY(check_attn_dims(B, N, Ci));
  GLF_TRY(check_ptr(P3, "P3"));
  GLF_TRY(check_ptr(Y, "Y"));
  GLF_TRY(check_ptr(lse, "lse"));
  GLF_TRY(check_scratch(scratch));
  GLF_TRY(check_device_sm100());
  WsAttn w;
  carve_ws_attn(B, N, Ci, false, scratch, &w);
  return flash_fwd(reinterpret_cast<const bf16*>(P3), reinterpret_cast<bf16*>(Y), lse, B, N, Ci, w.attn,
                   reinterpret_cast<cudaStream_t>(stream));
}

GLF_API int glf_attention_bwd(const void* P3, const void* Y, const void* dY, const float* lse, void* dP3,
                              float* bias_grad, int B, int N, int Ci, void* scratch, glf_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  GLF_TRY(check_attn_dims(B, N, Ci));
  GLF_TRY(check_ptr(P3, "P3"));
  GLF_TRY(check_ptr(Y, "Y"));
  GLF_TRY(check_ptr(dY, "dY"));
  GLF_TRY(check_ptr(lse, "lse"));
  GLF_TRY(check_ptr(dP3, "dP3"));
  if (bias_grad != nullptr) GLF_TRY(check_ptr(bias_grad, "bias_grad"));
  GLF_TRY(check_scratch(scratch));
  GLF_TRY(check_device_sm100());
  WsAttn w;
  carve_ws_attn(B, N, Ci, true, scratch, &w);
  ColTables cs;
  GLF_TRY(flash_bwd(reinterpret_cast<const bf16*>(P3), reinterpret_cast<const bf16*>(Y), reinterpret_cast<const bf16*>(dY),
                    lse, reinterpret_cast<bf16*>(dP3), w.delta, w.cs_t, w.cs_p, w.cs_g, w.cs_cap_rows, &cs, B, N, Ci,
                    w.attn, stream));
  if (bias_grad == nullptr) return 0;
  float* const db[3] = {bias_grad, bias_grad + Ci, bias_grad + 2 * Ci};
  return reduce_bias_grads(cs, Ci, w.red1, db, stream);
}

GLF_API size_t glf_attention_gaussian_scratch_bytes(int B, int N, int C, int Ci, int backward) {
  if (check_attn_dims(B, N, Ci) != 0 || check_attn_dims(B, N, C) != 0) return 0;
  WsAttn w;
  return carve_ws_attn(B, N, Ci, backward != 0, nullptr, &w, C);
}

GLF_API int glf_attention_gaussian_fwd(const void* X, const void* G, void* Y, float* lse, int B, int N, int C, int Ci,
                                       void* scratch, glf_stream_t stream) {
  GLF_TRY(check_attn_dims(B, N, Ci));
  GLF_TRY(check_attn_dims(B, N, C));
  GLF_TRY(check_ptr(X, "X"));
  GLF_TRY(check_ptr(G, "G"));
  GLF_TRY(check_ptr(Y, "Y"));
  GLF_TRY(check_ptr(lse, "lse"));
  GLF_TRY(check_scratch(scratch));
  GLF_TRY(check_device_sm100());
  WsAttn w;
  carve_ws_attn(B, N, Ci, false, scratch, &w, C);
  const AttnArgs a = attn_args_gaussian(reinterpret_cast<const bf16*>(X), reinterpret_cast<const bf16*>(G), nullptr,
                                        nullptr, nullptr, 0, 0, C, Ci);
  return attn_fwd(a, reinterpret_cast<bf16*>(Y), lse, B, N, w.attn, reinterpret_cast<cudaStream_t>(stream));
}

GLF_API int glf_attention_gaussian_bwd(const void* X, const void* G, const void* Y, const void* dY, const float* lse,
                                       void* dX, void* dG, float* bias_grad, int B, int N, int C, int Ci, void* scratch,
                                       glf_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  GLF_TRY(check_attn_dims(B, N, Ci));
  GLF_TRY(check_attn_dims(B, N, C));
  GLF_TRY(check_ptr(X, "X"));
  GLF_TRY(check_ptr(G, "G"));
  GLF_TRY(check_ptr(Y, "Y"));
  GLF_TRY(check_ptr(dY, "dY"));
  GLF_TRY(check_ptr(lse, "lse"));
  GLF_TRY(check_ptr(dX, "dX"));
  GLF_TRY(check_ptr(dG, "dG"));
  if (bias_grad != nullptr) GLF_TRY(check_ptr(bias_grad, "bias_grad"));
  GLF_TRY(check_scratch(scratch));
  GLF_TRY(check_device_sm100());
  WsAttn w;
  carve_ws_attn(B, N, Ci, true, scratch, &w, C);
  const AttnArgs a = attn_args_gaussian(reinterpret_cast<const bf16*>(X), reinterpret_cast<const bf16*>(G), w.dx2,
                                        w.dx2 + C, reinterpret_cast<bf16*>(dG), 2LL * C, Ci, C, Ci);
  ColTables cs;
  GLF_TRY(attn_bwd(a, reinterpret_cast<const bf16*>(Y), reinterpret_cast<const bf16*>(dY), lse, w.delta, w.cs_t, w.cs_p,
                   w.cs_g, w.cs_cap_rows, &cs, B, N, w.attn, stream));
  GLF_TRY(sum_halves(w.dx2, reinterpret_cast<bf16*>(dX), static_cast<long long>(B) * N, C, stream));
  if (bias_grad == nullptr) return 0;
  return reduce_bias_grads(cs, Ci, w.red1, &bias_grad, stream);
}

GLF_API int glf_bn_res_ln_fwd(int64_t rows, int C, const void* U, const void* X, const float* bn_a, const float* bn_b,
                              const float* ln_w, const float* ln_b, void* Z, int z_dtype, float* mu, float* r,
                              float eps, int accumulate, glf_stream_t stream) {
  GLF_TRY(check_device_sm100());
  GLF_TRY(check_ptr(X, "X"));
  GLF_TRY(check_ptr(Z, "Z"));
  if (rows <= 0) return set_error(GLF_ERR_INVALID, "empty input");
  return bn_res_ln_fwd(U, X, GLF_DTYPE_BF16, bn_a, bn_b, ln_w, ln_b, Z, z_dtype, mu, r, rows, C, eps, accumulate,
                       reinterpret_cast<cudaStream_t>(stream));
}

GLF_API int glf_bn_res_ln_bwd(int64_t rows, int C, const void* dZ, int dz_dtype, const void* U, const void* X,
                              const float* bn_a, const float* bn_b, const float* bn_mean, const float* bn_rstd,
                              const float* ln_w, const float* mu, const float* r, void* dV, float* part,
                              int* nblocks_out, glf_stream_t stream) {
  GLF_TRY(check_device_sm100());
  GLF_TRY(check_ptr(dZ, "dZ"));
  GLF_TRY(check_ptr(X, "X"));
  GLF_TRY(check_ptr(dV, "dV"));
  if (rows <= 0) return set_error(GLF_ERR_INVALID, "empty input");
  return bn_res_ln_bwd(dZ, dz_dtype, U, X, GLF_DTYPE_BF16, bn_a, bn_b, bn_mean, bn_rstd, ln_w, mu, r, dV, part, rows, C,
                       nblocks_out, reinterpret_cast<cudaStream_t>(stream));
}

GLF_API int glf_bn_res_ln_bwd_max_blocks(void) { return 148 * 2; }

// Pair forms with explicit operands (unit tests, roofline probe): index 0 = MGFM, 1 = MLFM.
GLF_API int glf_bn_res_ln_pair_fwd(int64_t rows, int C, const void* const* U, const void* const* X,
                                   const float* const* bn_a, const float* const* bn_b, const float* const* ln_w,
                                   const float* const* ln_b, void* Z, float* const* mu, float* const* r, float eps,
                                   int accumulate, glf_stream_t stream) {
  GLF_TRY(check_device_sm100());
  if (rows <= 0) return set_error(GLF_ERR_INVALID, "empty input");
  if (!ln_tma_supported(C)) return set_error(GLF_ERR_UNSUPPORTED, "fused LayerNorm pair needs C <= 256, C %% 8 == 0");
  GLF_TRY(check_ptr(Z, "Z"));
  for (int m = 0; m < 2; ++m) {
    GLF_TRY(check_ptr(U[m], "U"));
    GLF_TRY(check_ptr(X[m], "X"));
  }
  return ln_fwd_tma(2, reinterpret_cast<const bf16* const*>(U), reinterpret_cast<const bf16* const*>(X), bn_a, bn_b, ln_w,
                    ln_b, mu, r, reinterpret_cast<bf16*>(Z), rows, C, eps, accumulate,
                    reinterpret_cast<cudaStream_t>(stream));
}

GLF_API int glf_bn_res_ln_pair_bwd(int64_t rows, int C, const void* dZ, const void* const* U, const void* const* X,
                                   const float* const* bn_a, const float* const* bn_b, const float* const* bn_mean,
                                   const float* const* bn_rstd, const float* const* ln_w, const float* const* mu,
                                   const float* const* r, void* const* dV, float* const* part, int* nblocks_out,
                                   glf_stream_t stream) {
  GLF_TRY(check_device_sm100());
  if (rows <= 0) return set_error(GLF_ERR_INVALID, "empty input");
  if (!ln_tma_supported(C)) return set_error(GLF_ERR_UNSUPPORTED, "fused LayerNorm pair needs C <= 256, C %% 8 == 0");
  GLF_TRY(check_ptr(dZ, "dZ"));
  for (int m = 0; m < 2; ++m) {
    GLF_TRY(check_ptr(U[m], "U"));
    GLF_TRY(check_ptr(X[m], "X"));
    GLF_TRY(check_ptr(dV[m], "dV"));
    GLF_TRY(check_ptr(mu[m], "mu"));
    GLF_TRY(check_ptr(r[m], "r"));
  }
  return ln_bwd_tma(2, reinterpret_cast<const bf16*>(dZ), reinterpret_cast<const bf16* const*>(U),
                    reinterpret_cast<const bf16* const*>(X), bn_a, bn_b, ln_w, bn_mean, bn_rstd, mu, r,
                    reinterpret_cast<bf16* const*>(dV), part, rows, C, nblocks_out,
                    reinterpret_cast<cudaStream_t>(stream));
}

GLF_API size_t glf_cycle_loss_scratch_bytes(int T, int C, int n_starts) {
  if (T <= 0 || C <= 0 || n_starts <= 0) return 0;
  return cycle_loss_scratch_bytes(T, C, n_starts);
}

GLF_API int glf_cycle_loss(const float* feat, int T, int C, int target_region, int cyc_off, int chunk_size,
                           float temperature, int start, int step, int n_starts, int soft_label, float scale,
                           float* loss, float* dfeat, void* scratch, glf_stream_t stream) {
  GLF_TRY(check_device_sm100());
  GLF_TRY(check_ptr(feat, "feat"));
  GLF_TRY(check_ptr(loss, "loss"));
  GLF_TRY(check_ptr(dfeat, "dfeat"));
  GLF_TRY(check_ptr(scratch, "scratch"));
  return cycle_loss(feat, T, C, target_region, cyc_off, chunk_size, temperature, start, step, n_starts, soft_label,
                    scale, loss, dfeat, reinterpret_cast<float*>(scratch), reinterpret_cast<cudaStream_t>(stream));
}

GLF_API int glf_spatial_sums(const void* x, int dtype, int B, int C, int T, int64_t stride_b, int64_t stride_c,
                             int64_t stride_t, float* out, glf_stream_t stream) {
  GLF_TRY(check_device_sm100());
  if (x == nullptr || out == nullptr) return set_error(GLF_ERR_INVALID, "spatial_sums: NULL pointer");   // any element alignment
  return spatial_sums(x, dtype, B, C, T, stride_b, stride_c, stride_t, out, reinterpret_cast<cudaStream_t>(stream));
}

GLF_API int glf_transpose(const void* in, void* out, int batch, int R, int S, int in_dtype, int out_dtype,
                  glf_stream_t stream) {
  GLF_TRY(check_device_sm100());
  GLF_TRY(check_ptr(in, "in"));
  GLF_TRY(check_ptr(out, "out"));
  return transpose_cast(in, out, batch, R, S, in_dtype, out_dtype, reinterpret_cast<cudaStream_t>(stream));
}

}  // extern "C"
