// glf_api_f32.cu — GLF_PRECISION_F32X3: the mode='dot' forward/backward with fp32-exact products on tcgen05.
//
// Activations stay fp32 in HBM.  Before every product its operands are split into three bf16 limb planes
// (hi, mid, lo: x = l0 + l1 + l2 to 24 mantissa bits, split3_kernel) and the tcgen05 GEMM accumulates the six
// limb products of total order <= 2   (0,2) (2,0) (1,1) (0,1) (1,0) (0,0)   into one fp32 TMEM accumulator — the
// dropped terms are O(2^-24) relative.  Same kernels, same data flow as the bf16 path; this is the arm that meets the
// reference's fp32 tolerance (1e-4).  It is the precision arm, not the throughput arm.
#include "glf_internal.h"

namespace glf {

namespace {

struct Saved3 {
  float *Xf, *Uf, *bcat, *bn_mean, *bn_rstd, *bn_a, *bn_b, *ln_mu, *ln_r;
  bf16 *Xl, *Pl, *Ml, *Wpl, *wcat_l, *wcatT_l, *wz_l;
};
size_t carve_saved3(const Dims& m, void* base, Saved3* s) {
  Carver c(base);
  const size_t rows = m.rows, C = m.C, Ci = m.Ci, B = m.B;
  s->Xf = m.pack_x ? c.take<float>(rows * C) : nullptr;
  s->Xl = c.take<bf16>(3 * rows * C);
  s->Pl = c.take<bf16>(3 * rows * 3 * Ci);
  s->Uf = c.take<float>(rows * C);
  s->Ml = c.take<bf16>(3 * B * Ci * Ci);
  s->Wpl = c.take<bf16>(3 * B * C * Ci);
  s->wcat_l = c.take<bf16>(3 * 3 * Ci * C);
  s->wcatT_l = c.take<bf16>(3 * 3 * Ci * C);
  s->wz_l = c.take<bf16>(3 * C * Ci);
  s->bcat = c.take<float>(3 * Ci);
  s->bn_mean = c.take<float>(C);
  s->bn_rstd = c.take<float>(C);
  s->bn_a = c.take<float>(C);
  s->bn_b = c.take<float>(C);
  s->ln_mu = c.take<float>(rows);
  s->ln_r = c.take<float>(rows);
  return (c.off + 255) & ~static_cast<size_t>(255);
}

// Slab scratch of the fixed-order split reductions (GLF_DETERMINISTIC), last in ws: the largest need among the
// products that sum partials (M forward; dW', dWz, dWcat backward)
void carve_slab3(Carver& c, const Dims& m, bool backward, SplitSlab* s) {
  *s = SplitSlab{};
  if (!m.det) return;
  const int B = static_cast<int>(m.B), C = m.C, Ci = m.Ci, N = static_cast<int>(m.N), rows = static_cast<int>(m.rows);
  auto t = [](long long n) { return (n + 127) / 128; };
  long long need = 0;
  auto take = [&need](long long v) { need = v > need ? v : need; };
  if (!backward) {
    take(slab_need(Ci, Ci, B, N, pick_split(B * t(Ci) * t(Ci), N), false, false));
  } else {
    take(slab_need(C, Ci, B, N, pick_split(B * t(C) * t(Ci), N), false, false));
    take(slab_need(C, Ci, B, Ci, 1, true, false));
    take(slab_need(3 * Ci, C, 1, rows, pick_split(t(3 * Ci) * t(C), rows), false, false));
  }
  s->on = true;
  s->floats = need;
  if (need > 0) s->p = c.take<float>(static_cast<size_t>(need));
}

struct WsF3 { float *wcat_f, *wcatT_f, *Pf, *Mf, *Wpf, *cs; void* saved_fallback; SplitSlab det; };
size_t carve_wsf3(const Dims& m, void* base, WsF3* w, size_t saved_bytes) {
  Carver c(base);
  const size_t rows = m.rows, C = m.C, Ci = m.Ci, B = m.B;
  w->wcat_f = c.take<float>(3 * Ci * C);
  w->wcatT_f = c.take<float>(3 * Ci * C);
  w->Pf = c.take<float>(rows * 3 * Ci);
  w->Mf = c.take<float>(B * Ci * Ci);
  w->Wpf = c.take<float>(B * C * Ci);
  w->cs = c.take<float>(static_cast<size_t>(colstats_f32_blocks(m.rows)) * 2 * C);
  w->saved_fallback = c.take<uint8_t>(saved_bytes);
  carve_slab3(c, m, false, &w->det);
  return (c.off + 255) & ~static_cast<size_t>(255);
}

struct WsB3 {
  float *dZf, *dVf, *dUf, *dPf, *dWpf, *dMf, *dXf, *part_ln, *k1, *k2, *k3, *cs, *dwcat;
  bf16 *dUl, *dPl, *dWpl, *dMl;
  SplitSlab det;
};
size_t carve_wsb3(const glf_desc* d, const Dims& m, void* base, WsB3* w) {
  Carver c(base);
  const size_t rows = m.rows, C = m.C, Ci = m.Ci, B = m.B;
  const bool dz_f32_tokens = d->dz_layout == GLF_LAYOUT_TOKEN && d->io_dtype == GLF_DTYPE_F32;   // read in place
  w->dZf = dz_f32_tokens ? nullptr : c.take<float>(rows * C);
  w->dVf = c.take<float>(rows * C);
  w->dUf = c.take<float>(rows * C);
  w->dUl = c.take<bf16>(3 * rows * C);
  w->dPf = c.take<float>(rows * 3 * Ci);
  w->dPl = c.take<bf16>(3 * rows * 3 * Ci);
  w->dWpf = c.take<float>(B * C * Ci);
  w->dWpl = c.take<bf16>(3 * B * C * Ci);
  w->dMf = c.take<float>(B * Ci * Ci);
  w->dMl = c.take<bf16>(3 * B * Ci * Ci);
  w->dXf = m.pack_x ? c.take<float>(rows * C) : nullptr;
  w->part_ln = c.take<float>(static_cast<size_t>(bn_res_ln_bwd_blocks(m.rows, m.C)) * 4 * C);
  w->k1 = c.take<float>(C);
  w->k2 = c.take<float>(C);
  w->k3 = c.take<float>(C);
  w->cs = c.take<float>(static_cast<size_t>(colstats_f32_blocks(m.rows)) * 2 * 3 * Ci);
  w->dwcat = c.take<float>(3 * Ci * C);
  carve_slab3(c, m, true, &w->det);
  return (c.off + 255) & ~static_cast<size_t>(255);
}

void six_pairs(GemmArgs& g) {
  static const int pa[6] = {0, 2, 1, 0, 1, 0};
  static const int pb[6] = {2, 0, 1, 1, 0, 0};
  g.npairs = 6;
  for (int i = 0; i < 6; ++i) { g.pairA[i] = pa[i]; g.pairB[i] = pb[i]; }
}
}  // namespace

int tpavi_sizes_f32x3(const glf_desc* d, const Dims& m, glf_sizes* out) {
  Saved3 s; WsF3 wf; WsB3 wb;
  out->saved_bytes = carve_saved3(m, nullptr, &s);
  out->ws_fwd_bytes = carve_wsf3(m, nullptr, &wf, out->saved_bytes);
  out->ws_bwd_bytes = carve_wsb3(d, m, nullptr, &wb);
  return 0;
}

int tpavi_fwd_f32x3(const glf_desc* d, const Dims& m, const void* x, const glf_weights* w, void* z, void* saved,
                    void* ws, cudaStream_t stream) {
  Saved3 s; WsF3 wf;
  const size_t saved_bytes = carve_saved3(m, nullptr, &s);
  carve_wsf3(m, ws, &wf, saved_bytes);
  carve_saved3(m, saved ? saved : wf.saved_fallback, &s);
  const int C = m.C, Ci = m.Ci, N = static_cast<int>(m.N), B = static_cast<int>(m.B), rows = static_cast<int>(m.rows);
  const long long pX = static_cast<long long>(rows) * C, pP = static_cast<long long>(rows) * 3 * Ci;
  const long long pW = 3LL * Ci * C, pWz = static_cast<long long>(C) * Ci;
  const long long CiCi = static_cast<long long>(Ci) * Ci, CCi = pWz;
  const long long pM = B * CiCi, pWp = B * CCi;
  const long long seqP = static_cast<long long>(N) * 3 * Ci;

  GLF_TRY(prep_weights_f32(w, C, Ci, wf.wcat_f, wf.wcatT_f, s.bcat, stream));
  GLF_TRY(split3(wf.wcat_f, s.wcat_l, pW, stream));
  GLF_TRY(split3(wf.wcatT_f, s.wcatT_l, pW, stream));
  GLF_TRY(split3(w->wz_w, s.wz_l, pWz, stream));
  const float* Xf = reinterpret_cast<const float*>(x);
  if (m.pack_x) {
    GLF_TRY(pack_tokens(m, x, d->io_dtype, d->x_layout == GLF_LAYOUT_NCTHW, s.Xf, GLF_DTYPE_F32, stream));
    Xf = s.Xf;
  }
  GLF_TRY(split3(Xf, s.Xl, pX, stream));
  {  // P = X Wcat^T + bcat
    GemmArgs g;
    g.A = opnd(s.Xl, 0, C, 0, pX);
    g.B = opnd(s.wcat_l, 0, C, 0, pW);
    six_pairs(g);
    g.M = rows; g.N = 3 * Ci; g.K = C;
    g.bias = s.bcat;
    g.out_kind = 1;
    g.D = wf.Pf; g.ldd = 3 * Ci;
    GLF_TRY(gemm(g, stream));
  }
  GLF_TRY(split3(wf.Pf, s.Pl, pP, stream));
  {  // M_b = Phi_b^T G_b / N
    GemmArgs g;
    g.A = opnd(s.Pl + Ci, 1, 3 * Ci, seqP, pP);
    g.B = opnd(s.Pl + 2 * Ci, 1, 3 * Ci, seqP, pP);
    six_pairs(g);
    g.M = Ci; g.N = Ci; g.K = N; g.batch = B;
    g.alpha = 1.f / static_cast<float>(N);
    g.ldd = Ci; g.strideD = CiCi;
    g.D = wf.Mf;
    g.det = wf.det;
    g.split_k = pick_split(static_cast<long long>(B) * ((Ci + 127) / 128) * ((Ci + 127) / 128), N);
    if (g.split_k > 1) {
      GLF_TRY(check_cuda(cudaMemsetAsync(wf.Mf, 0, sizeof(float) * pM, stream), "memset M"));
      g.out_kind = 2;
    } else {
      g.out_kind = 1;
    }
    GLF_TRY(gemm(g, stream));
  }
  GLF_TRY(split3(wf.Mf, s.Ml, pM, stream));
  {  // W'_b = Wz M_b^T
    GemmArgs g;
    g.A = opnd(s.wz_l, 0, Ci, 0, pWz);
    g.B = opnd(s.Ml, 0, Ci, CiCi, pM);
    six_pairs(g);
    g.M = C; g.N = Ci; g.K = Ci; g.batch = B;
    g.out_kind = 1;
    g.D = wf.Wpf; g.ldd = Ci; g.strideD = CCi;
    GLF_TRY(gemm(g, stream));
  }
  GLF_TRY(split3(wf.Wpf, s.Wpl, pWp, stream));
  {  // U_b = Theta_b W'_b^T + bz
    GemmArgs g;
    g.A = opnd(s.Pl, 0, 3 * Ci, seqP, pP);
    g.B = opnd(s.Wpl, 0, Ci, CCi, pWp);
    six_pairs(g);
    g.M = N; g.N = C; g.K = Ci; g.batch = B;
    g.bias = w->wz_b;
    g.out_kind = 1;
    g.D = s.Uf; g.ldd = C; g.strideD = static_cast<long long>(N) * C;
    GLF_TRY(gemm(g, stream));
  }
  int np = 0;
  if (d->training && d->bn_layer) {
    GLF_TRY(colstats_f32(s.Uf, wf.cs, m.rows, C, stream));
    np = colstats_f32_blocks(m.rows);
  }
  GLF_TRY(bn_finalize(wf.cs, np, C, static_cast<double>(m.rows), d, w, nullptr, s.bn_mean, s.bn_rstd, s.bn_a, s.bn_b, stream));
  GLF_TRY(bn_res_ln_fwd(s.Uf, Xf, GLF_DTYPE_F32, s.bn_a, s.bn_b, w->ln_w, w->ln_b, z, d->io_dtype, s.ln_mu, s.ln_r,
                        m.rows, C, d->eps_ln, d->accumulate, stream));
  return 0;
}

int tpavi_bwd_f32x3(const glf_desc* d, const Dims& m, const void* dz, const void* x, const glf_weights* w,
                    const void* saved, void* dx, const glf_grads* g_, void* ws, cudaStream_t stream) {
  Saved3 s; WsB3 wb;
  carve_saved3(m, const_cast<void*>(saved), &s);
  carve_wsb3(d, m, ws, &wb);
  const int C = m.C, Ci = m.Ci, N = static_cast<int>(m.N), B = static_cast<int>(m.B), rows = static_cast<int>(m.rows);
  const long long pX = static_cast<long long>(rows) * C, pP = static_cast<long long>(rows) * 3 * Ci;
  const long long pW = 3LL * Ci * C, pWz = static_cast<long long>(C) * Ci;
  const long long CiCi = static_cast<long long>(Ci) * Ci, CCi = pWz;
  const long long pM = B * CiCi, pWp = B * CCi;
  const long long seqP = static_cast<long long>(N) * 3 * Ci;
  const float* Xf = m.pack_x ? s.Xf : reinterpret_cast<const float*>(x);

  const void* dZ = dz;
  int dz_dtype = d->io_dtype;
  if (m.pack_dz) {
    GLF_TRY(pack_tokens(m, dz, d->io_dtype, /*ncthw=*/true, wb.dZf, GLF_DTYPE_F32, stream));
    dZ = wb.dZf;
    dz_dtype = GLF_DTYPE_F32;
  }
  int nb = 0;
  GLF_TRY(bn_res_ln_bwd(dZ, dz_dtype, s.Uf, Xf, GLF_DTYPE_F32, s.bn_a, s.bn_b, s.bn_mean, s.bn_rstd, w->ln_w, s.ln_mu,
                        s.ln_r, wb.dVf, wb.part_ln, m.rows, C, &nb, stream));
  GLF_TRY(bn_bwd_finalize(wb.part_ln, nb, C, static_cast<double>(m.rows), d, w, s.bn_mean, s.bn_rstd, g_, wb.k1, wb.k2,
                          wb.k3, stream));
  const float* dUf = wb.dVf;
  if (d->bn_layer) {
    GLF_TRY(bn_bwd_apply(wb.dVf, s.Uf, GLF_DTYPE_F32, wb.k1, wb.k2, wb.k3, wb.dUf, m.rows, C, stream));
    dUf = wb.dUf;
  }
  GLF_TRY(split3(dUf, wb.dUl, pX, stream));
  {  // dTheta_b = dU_b W'_b
    GemmArgs g;
    g.A = opnd(wb.dUl, 0, C, static_cast<long long>(N) * C, pX);
    g.B = opnd(s.Wpl, 1, Ci, CCi, pWp);
    six_pairs(g);
    g.M = N; g.N = Ci; g.K = C; g.batch = B;
    g.out_kind = 1;
    g.D = wb.dPf; g.ldd = 3 * Ci; g.strideD = seqP;
    GLF_TRY(gemm(g, stream));
  }
  {  // dW'_b = dU_b^T Theta_b
    GemmArgs g;
    g.A = opnd(wb.dUl, 1, C, static_cast<long long>(N) * C, pX);
    g.B = opnd(s.Pl, 1, 3 * Ci, seqP, pP);
    six_pairs(g);
    g.M = C; g.N = Ci; g.K = N; g.batch = B;
    g.ldd = Ci; g.strideD = CCi;
    g.D = wb.dWpf;
    g.det = wb.det;
    g.split_k = pick_split(static_cast<long long>(B) * ((C + 127) / 128) * ((Ci + 127) / 128), N);
    if (g.split_k > 1) {
      GLF_TRY(check_cuda(cudaMemsetAsync(wb.dWpf, 0, sizeof(float) * pWp, stream), "memset dW'"));
      g.out_kind = 2;
    } else {
      g.out_kind = 1;
    }
    GLF_TRY(gemm(g, stream));
  }
  GLF_TRY(split3(wb.dWpf, wb.dWpl, pWp, stream));
  GLF_TRY(check_cuda(cudaMemsetAsync(g_->wz_w, 0, sizeof(float) * CCi, stream), "memset dWz"));
  {  // dWz = sum_b dW'_b M_b
    GemmArgs g;
    g.A = opnd(wb.dWpl, 0, Ci, CCi, pWp);
    g.B = opnd(s.Ml, 1, Ci, CiCi, pM);
    six_pairs(g);
    g.M = C; g.N = Ci; g.K = Ci; g.batch = B;
    g.out_kind = 2;
    g.det = wb.det;
    g.D = g_->wz_w; g.ldd = Ci; g.strideD = 0;
    GLF_TRY(gemm(g, stream));
  }
  {  // dM_b = dW'_b^T Wz
    GemmArgs g;
    g.A = opnd(wb.dWpl, 1, Ci, CCi, pWp);
    g.B = opnd(s.wz_l, 1, Ci, 0, pWz);
    six_pairs(g);
    g.M = Ci; g.N = Ci; g.K = C; g.batch = B;
    g.out_kind = 1;
    g.D = wb.dMf; g.ldd = Ci; g.strideD = CiCi;
    GLF_TRY(gemm(g, stream));
  }
  GLF_TRY(split3(wb.dMf, wb.dMl, pM, stream));
  {  // dPhi_b = G_b dM_b^T / N
    GemmArgs g;
    g.A = opnd(s.Pl + 2 * Ci, 0, 3 * Ci, seqP, pP);
    g.B = opnd(wb.dMl, 0, Ci, CiCi, pM);
    six_pairs(g);
    g.M = N; g.N = Ci; g.K = Ci; g.batch = B;
    g.alpha = 1.f / static_cast<float>(N);
    g.out_kind = 1;
    g.D = wb.dPf + Ci; g.ldd = 3 * Ci; g.strideD = seqP;
    GLF_TRY(gemm(g, stream));
  }
  {  // dG_b = Phi_b dM_b / N
    GemmArgs g;
    g.A = opnd(s.Pl + Ci, 0, 3 * Ci, seqP, pP);
    g.B = opnd(wb.dMl, 1, Ci, CiCi, pM);
    six_pairs(g);
    g.M = N; g.N = Ci; g.K = Ci; g.batch = B;
    g.alpha = 1.f / static_cast<float>(N);
    g.out_kind = 1;
    g.D = wb.dPf + 2 * Ci; g.ldd = 3 * Ci; g.strideD = seqP;
    GLF_TRY(gemm(g, stream));
  }
  GLF_TRY(split3(wb.dPf, wb.dPl, pP, stream));
  {  // bias gradients = column sums of dP
    GLF_TRY(colstats_f32(wb.dPf, wb.cs, m.rows, 3 * Ci, stream));
    const int np = colstats_f32_blocks(m.rows);
    GLF_TRY(reduce_partials3(wb.cs, wb.cs + Ci, wb.cs + 2 * Ci, np, 2LL * 3 * Ci, Ci, g_->theta_b, g_->phi_b, g_->g_b,
                             stream));
  }
  GLF_TRY(check_cuda(cudaMemsetAsync(wb.dwcat, 0, sizeof(float) * pW, stream), "memset dWcat"));
  {  // dWcat = dP^T X
    GemmArgs g;
    g.A = opnd(wb.dPl, 1, 3 * Ci, 0, pP);
    g.B = opnd(s.Xl, 1, C, 0, pX);
    six_pairs(g);
    g.M = 3 * Ci; g.N = C; g.K = rows;
    g.out_kind = 2;
    g.det = wb.det;
    g.D = wb.dwcat; g.ldd = C;
    g.split_k = pick_split(static_cast<long long>((3 * Ci + 127) / 128) * ((C + 127) / 128), rows);
    GLF_TRY(gemm(g, stream));
  }
  GLF_TRY(scatter_proj_grads(wb.dwcat, g_, C, Ci, false, stream));
  {  // dX = dV + dP Wcat : the output is initialised with dV and the product is accumulated onto it (fp32 red.add)
    float* dXf = m.pack_x ? wb.dXf : reinterpret_cast<float*>(dx);
    GLF_TRY(check_cuda(cudaMemcpyAsync(dXf, wb.dVf, sizeof(float) * pX, cudaMemcpyDeviceToDevice, stream), "copy dV"));
    GemmArgs g;
    g.A = opnd(wb.dPl, 0, 3 * Ci, 0, pP);
    g.B = opnd(s.wcatT_l, 0, 3 * Ci, 0, pW);
    six_pairs(g);
    g.M = rows; g.N = C; g.K = 3 * Ci;
    g.out_kind = 2;
    g.det = wb.det;
    g.D = dXf; g.ldd = C;
    GLF_TRY(gemm(g, stream));
    if (m.pack_x)
      GLF_TRY(unpack_tokens(m, dXf, GLF_DTYPE_F32, dx, d->x_layout == GLF_LAYOUT_NCTHW, d->io_dtype, stream));
  }
  return 0;
}

}  // namespace glf
