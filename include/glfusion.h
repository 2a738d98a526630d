/* glfusion.h — C ABI of libglf_sm100a.so: the B200-native GL-Fusion cross-view fusion hot path.
 *
 * Reference being replaced (R = xmed-lab/GL-Fusion, GLfusion/):
 *   - TPAVIModule.forward            R/models/ours.py:845-917  (dup R/models/TPAVI.py:86-155)   -> glf_tpavi_fwd
 *   - its autograd backward          (implicit in the reference)                                 -> glf_tpavi_bwd
 *   - gate + view concat             R/models/ours.py:1802-1820, 1826-1827                       -> glf_gate_concat_fwd
 *   - their backward                 (implicit)                                                  -> glf_gate_concat_bwd
 *   - MGFM + MLFM sum, .contiguous() R/models/ours.py:1833-1837                                  -> glf_tpavi_fwd (accumulate flag)
 * The reference has no FFI layer for this path (pure Python nn.Module, SURVEY.md §8b); this header is the
 * boundary a maintainer binds with ctypes (see INTEGRATION.md).
 *
 * Contract
 *   - plain pointers and sizes only; every pointer is DEVICE memory on the current CUDA device unless noted;
 *   - the caller allocates everything (outputs, saved-for-backward blob, workspace); the library never
 *     allocates, frees or synchronises, and enqueues all work on the given stream (CUDA-graph capturable);
 *   - return 0 on success, <0 on error; message via glf_last_error() (thread local); no fallback paths:
 *     unsupported configurations and non-sm_100 devices are errors;
 *   - re-entrant: no global mutable state besides a per-process cache of the driver entry point.
 */
#ifndef GLFUSION_H_
#define GLFUSION_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GLF_VERSION 100

#if defined(__GNUC__)
#define GLF_API __attribute__((visibility("default")))
#else
#define GLF_API
#endif

typedef void* glf_stream_t; /* cudaStream_t */

/* TPAVIModule(mode=...)  ours.py:869-900.  GLF_MODE_GAUSSIAN: f = X X^T on the block input itself (theta / phi take no
 * part; their glf_weights / glf_grads pointers are ignored and may be NULL), y = softmax(f) g(x). */
enum { GLF_MODE_DOT = 0, GLF_MODE_EMBEDDED = 1, GLF_MODE_GAUSSIAN = 2 };
/* I/O dtypes of the activations a caller hands over.  GLF_DTYPE_F16 is an I/O type only (torch.autocast's default):
 * the boundary kernels convert it to bf16 where they read it and round to fp16 where they write; everything between
 * (tensor-core operands, statistics) is bf16 / fp32 as for bf16 input.  fp16 stores round to nearest, so a value
 * beyond the fp16 range becomes +-inf (what torch.amp.GradScaler looks for), never a clamped 65504. */
enum { GLF_DTYPE_BF16 = 0, GLF_DTYPE_F32 = 1, GLF_DTYPE_F16 = 2 };
enum { GLF_LAYOUT_NCTHW = 0, GLF_LAYOUT_TOKEN = 1 };      /* [B,C,T,H,W] contiguous  |  [B,T,H,W,C] contiguous */
enum { GLF_PRECISION_BF16 = 0, GLF_PRECISION_F32X3 = 1 }; /* tensor-core operand precision */
/* Storage dtype of the glf_weights / glf_grads tensors (glf_desc.reserved[3]); 0 is fp32, the default. */
enum { GLF_PARAMS_F32 = 0, GLF_PARAMS_BF16 = 1, GLF_PARAMS_F16 = 2 };

enum {
  GLF_OK = 0,
  GLF_ERR_INVALID = -1,     /* bad argument / unsupported shape */
  GLF_ERR_UNSUPPORTED = -2, /* feature not available (e.g. mode='concatenate', dimension != 3) */
  GLF_ERR_DEVICE = -3,      /* not an sm_100 device, or CUDA error */
  GLF_ERR_WORKSPACE = -4    /* caller-provided blob too small / misaligned */
};

/* Problem descriptor: x is [B, C, T, H, W]; N = T*H*W tokens per sequence; Ci = inter_channels (C/2 by default). */
typedef struct glf_desc {
  int32_t B, T, H, W, C, Ci;
  int32_t mode;       /* GLF_MODE_* */
  int32_t io_dtype;   /* dtype of x, z, dz, dx                         GLF_DTYPE_* */
  int32_t x_layout;   /* physical layout of x and dx                   GLF_LAYOUT_* */
  int32_t dz_layout;  /* physical layout of dz (z itself is always GLF_LAYOUT_TOKEN, like the reference's
                         permuted LayerNorm output, ours.py:913-915) */
  int32_t precision;  /* GLF_PRECISION_* (GLF_PRECISION_F32X3: mode='dot' only; fp32 or bf16 io_dtype, not fp16) */
  int32_t training;   /* BatchNorm3d uses batch statistics and updates running stats (ours.py:822-825) */
  int32_t bn_layer;   /* 1: W_z = conv + BN ; 0: W_z = conv only (ours.py:829-833) */
  int32_t accumulate; /* fwd: z += result instead of z = result (fuses f4_global + f4_local, ours.py:1834) */
  float eps_bn, eps_ln, momentum;
  int32_t reserved[4]; /* reserved[0] = 1: "deferred LayerNorm" — glf_tpavi_fwd stops after the BatchNorm statistics and
                          glf_tpavi_bwd starts after the LayerNorm backward; the caller runs that stage for MGFM and
                          MLFM together with glf_fusion_ln_fwd / glf_fusion_ln_bwd (below).
                          reserved[1]: algorithm of mode='dot' (both are exact reassociations of ours.py:881-902):
                          0 = the library chooses (Gram form when N >= 5 C), 1 = token-space form (theta/phi/g formed
                          per token), 2 = Gram form (S = X~^T X~ per sequence, channel-space products only).
                          reserved[1] | GLF_DETERMINISTIC: bitwise run-to-run reproducible results (below).
                          reserved[2]: dtype of z / z_global / dz of the fused LayerNorm pass (GLF_DTYPE_BF16 or F16).
                          reserved[3]: GLF_PARAMS_* — element type of every glf_weights / glf_grads tensor, the running
                          statistics included (bn_num_batches_tracked stays int64).  With GLF_PARAMS_BF16 / F16 the block
                          computes exactly what fp32 parameters holding the same values compute: one launch per block
                          converts them to an fp32 copy inside `saved` (inside ws when saved is NULL) forward, and one
                          rounds the fp32 gradients to nearest into glf_grads backward (fp16 overflow: +-inf); the running
                          statistics are updated in place, rounded once.  GLF_PRECISION_F32X3 needs GLF_PARAMS_F32. */
} glf_desc;

/* Flag ORed into glf_desc.reserved[1] (the low byte keeps the mode='dot' algorithm): every product that would sum the
 * partial results of several K slices or batch entries with fp32 atomics instead stores each partial into its own slab
 * of ws and sums the slabs in a fixed order, so glf_tpavi_fwd / glf_tpavi_bwd give bitwise identical outputs and
 * gradients from run to run (same descriptor, device and build).  Everything else already reduces in a fixed order.
 * glf_tpavi_sizes counts the slabs in ws_fwd_bytes / ws_bwd_bytes only when the flag is set and a split occurs; the
 * glf_fusion_ln_* entry points accept the flag and ignore it. */
#define GLF_DETERMINISTIC 0x100

/* Master parameters, same shapes as the reference state_dict (SURVEY.md §8b): fp32, or the bf16 / fp16 element type
 * glf_desc.reserved[3] names (the pointers are then read as that type). */
typedef struct glf_weights {
  const float* theta_w; /* [Ci, C]   theta.weight[Ci,C,1,1,1] */
  const float* theta_b; /* [Ci] */
  const float* phi_w;   /* [Ci, C] */
  const float* phi_b;   /* [Ci] */
  const float* g_w;     /* [Ci, C] */
  const float* g_b;     /* [Ci] */
  const float* wz_w;    /* [C, Ci]   W_z.0.weight (or W_z.weight when bn_layer=0) */
  const float* wz_b;    /* [C] */
  const float* bn_w;    /* [C]       W_z.1.weight  (unused when bn_layer=0) */
  const float* bn_b;    /* [C]       W_z.1.bias */
  float* bn_running_mean;          /* [C]  updated in place when training */
  float* bn_running_var;           /* [C] */
  int64_t* bn_num_batches_tracked; /* [1] */
  const float* ln_w; /* [C]  norm_layer.weight */
  const float* ln_b; /* [C]  norm_layer.bias */
} glf_weights;

/* Gradients in the parameters' element type (glf_desc.reserved[3]), written (not accumulated) by glf_tpavi_bwd. */
typedef struct glf_grads {
  float* theta_w; float* theta_b;
  float* phi_w;   float* phi_b;
  float* g_w;     float* g_b;
  float* wz_w;    float* wz_b;
  float* bn_w;    float* bn_b;
  float* ln_w;    float* ln_b;
} glf_grads;

typedef struct glf_sizes {
  size_t saved_bytes;  /* blob written by fwd, read by bwd (activations kept for backward) */
  size_t ws_fwd_bytes; /* scratch for fwd */
  size_t ws_bwd_bytes; /* scratch for bwd */
} glf_sizes;

GLF_API int glf_version(void);
GLF_API const char* glf_last_error(void);

/* Sizes of the caller-allocated blobs for a descriptor (256-byte aligned pointers required). */
GLF_API int glf_tpavi_sizes(const glf_desc* d, glf_sizes* out);

/* z = LayerNorm(BN(W_z(attn(theta(x), phi(x), g(x)))) + x).   z: [B,T,H,W,C] contiguous, io_dtype.
 * `saved` may be NULL when no backward will follow (inference); then nothing is kept. */
GLF_API int glf_tpavi_fwd(const glf_desc* d, const void* x, const glf_weights* w, void* z, void* saved, void* ws,
                  glf_stream_t stream);

/* dx (layout/dtype of x) and all parameter gradients from dz.  `x` is the forward input again. */
GLF_API int glf_tpavi_bwd(const glf_desc* d, const void* dz, const void* x, const glf_weights* w, const void* saved,
                  void* dx, const glf_grads* g, void* ws, glf_stream_t stream);

/* Fused call site (ours.py:1821-1834): out = MGFM(x_g) + MLFM(x_l).  The two blocks' residual + LayerNorm stages are
 * HBM-bound and share a tensor each way (the output sum forward, dz backward), so they run as ONE pass:
 *   1. glf_tpavi_fwd(d, x_g, w_g, z, saved_g, ws)  and  glf_tpavi_fwd(d, x_l, w_l, z, saved_l, ws)  with
 *      d->reserved[0] = 1  (everything up to the BatchNorm statistics; z is not written),
 *   2. glf_fusion_ln_fwd: z (+)= LN_g(BN_g(U_g) + x_g) + LN_l(BN_l(U_l) + x_l)   (d->accumulate honoured),
 *   3. backward: glf_fusion_ln_bwd fills dV / the per-channel partials inside ws_g and ws_l (each sized
 *      ws_bwd_bytes), then glf_tpavi_bwd(d, dz, x_g, ..., ws_g) and glf_tpavi_bwd(d, dz, x_l, ..., ws_l) with
 *      d->reserved[0] = 1 continue from there.
 * Requirements (glf_fusion_ln_supported returns 1): bf16 token-major x, dz token-major, GLF_PRECISION_BF16, C <= 2048
 * (C <= 256: one bulk-copy pass each way; wider rows: one sliced-row pass forward, the two blocks' backward passes back
 * to back).  z, z_global and dz are bf16, or fp16 with d->reserved[2] = GLF_DTYPE_F16. */
GLF_API int glf_fusion_ln_supported(const glf_desc* d);
GLF_API int glf_fusion_ln_fwd(const glf_desc* d, const void* xg, const void* xl, const glf_weights* wg,
                      const glf_weights* wl, void* z, void* saved_g, void* saved_l, glf_stream_t stream);
/* Same pass, also storing the MGFM part on its own: z_global = LN_g(BN_g(U_g) + x_g) (token-major, dtype of z) —
 * f4_global_fusion of R/models/ours.py:1823, which the trainer's cycle-consistency pass consumes (R/main.py:211-235);
 * the MLFM part is z - z_global.  z_global == NULL is glf_fusion_ln_fwd. */
GLF_API int glf_fusion_ln_fwd_parts(const glf_desc* d, const void* xg, const void* xl, const glf_weights* wg,
                            const glf_weights* wl, void* z, void* z_global, void* saved_g, void* saved_l,
                            glf_stream_t stream);
GLF_API int glf_fusion_ln_bwd(const glf_desc* d, const void* dz, const void* xg, const void* xl, const glf_weights* wg,
                      const glf_weights* wl, const void* saved_g, const void* saved_l, void* ws_g, void* ws_l,
                      glf_stream_t stream);
/* The same backward pass with dz given PER VIEW, as the dict-keyed call site receives it (one [B, C, h, w] gradient per
 * view, ours.py:1833-1837): dz_views[v] points at view v's gradient stored as rows of C channels (channels_last, or a
 * view of a token-major stack): element (b, c, t) at b * dz_stride_b[v] + t * C + c, v < d->T.  The pass reads each
 * view where it lies; nothing is gathered first.  Needs h*w to be a multiple of the pass's 28-row tile
 * (glf_fusion_ln_bwd_views_supported returns 1); dz_views == NULL is glf_fusion_ln_bwd. */
GLF_API int glf_fusion_ln_bwd_views_supported(const glf_desc* d);
GLF_API int glf_fusion_ln_bwd_views(const glf_desc* d, const void* dz, const void* const* dz_views,
                            const int64_t* dz_stride_b, const void* xg, const void* xl, const glf_weights* wg,
                            const glf_weights* wl, const void* saved_g, const void* saved_l, void* ws_g, void* ws_l,
                            glf_stream_t stream);

/* Gate + view concat (ours.py:1802-1820,1826-1827).
 *   f4[v]  : [B, C, h, w]  io_dtype (bf16, fp16 or fp32), NCHW contiguous, v < V (host array of V device pointers, V <= 8)
 *   cls[v] : [B, ncls, h, w] fp32 logits of classifier[view];  ctr[v] : [B, 1, h, w] fp32 logits of centerness[view]
 *   xg, xl : [B, V*h*w, C] token-major (view-major token order, i.e. T = V), x_dtype (bf16, or fp32 for the
 *            GLF_PRECISION_F32X3 arm)                                                 — MGFM / MLFM inputs
 *   gate   : [B, V, h, w] fp32, a = sigmoid(weight * max_c sigmoid(cls) * sigmoid(ctr))   (kept for backward) */
GLF_API int glf_gate_concat_fwd(int B, int C, int V, int h, int w, int ncls, float weight, int io_dtype, int x_dtype,
                        const void* const* f4, const float* const* cls, const float* const* ctr, void* xg, void* xl,
                        float* gate, glf_stream_t stream);

/* df4[v] = dxg[:, v] + gate * dxl[:, v]  (NCHW, io_dtype);  dcls[v], dctr[v] fp32 logit gradients.
 * scratch: caller-allocated, glf_gate_concat_bwd_scratch_bytes(...) bytes (per-channel-tile partials of the gate
 * gradient, reduced in a fixed order). */
GLF_API size_t glf_gate_concat_bwd_scratch_bytes(int B, int C, int V, int h, int w);
GLF_API int glf_gate_concat_bwd(int B, int C, int V, int h, int w, int ncls, float weight, int io_dtype, int x_dtype,
                        const void* const* f4, const float* const* cls, const float* const* ctr, const float* gate,
                        const void* dxg, const void* dxl, void* const* df4, float* const* dcls, float* const* dctr,
                        void* scratch, glf_stream_t stream);

/* The same two steps for CHANNELS-LAST views (SURVEY.md section 8 f1: backbones / heads run channels_last, so
 * f4[v] arrives as rows of C channels — element (b, c, t) at b*stride_b[v] + t*stride_t[v] + c, t = y*w + x): no
 * transposition is left, gate + concat is a row kernel, and df4[v] is written in the layout dstride_b / dstride_t
 * describe (channels-last again, so the conv backward that consumes it stays channels_last).  io_dtype: dtype of f4 /
 * df4; xg / xl / dxg / dxl bf16 token-major; cls / ctr logits and their gradients fp32 NCHW as above; rows must be
 * 16-byte aligned.  scratch: glf_gate_concat_bwd_scratch_bytes bytes. */
GLF_API int glf_gate_concat_cl_fwd(int B, int C, int V, int h, int w, int ncls, float weight, int io_dtype,
                           const void* const* f4, const int64_t* stride_b, const int64_t* stride_t,
                           const float* const* cls, const float* const* ctr, void* xg, void* xl, float* gate,
                           glf_stream_t stream);
GLF_API int glf_gate_concat_cl_bwd(int B, int C, int V, int h, int w, int ncls, float weight, int io_dtype,
                           const void* const* f4, const int64_t* stride_b, const int64_t* stride_t,
                           const float* const* cls, const float* const* ctr, const float* gate, const void* dxg,
                           const void* dxl, void* const* df4, const int64_t* dstride_b, const int64_t* dstride_t,
                           float* const* dcls, float* const* dctr, void* scratch, glf_stream_t stream);

/* The dict-keyed call site's backward: V per-view gradients ([B, C, h, w]; element strides of batch / channel / the
 * collapsed h*w axis given per view, one of the last two must be 1: NCHW or channels-last) gathered into ONE
 * token-major [B, V, T, C] bf16 buffer, the transposition ours.py:1819-1820 performs forward (permute + cat); src_dtype
 * bf16, fp16 or fp32 (converted on the way).  A stride of 0 is allowed (a broadcast gradient).  A NULL
 * entry of `src` (a view whose output received no gradient) is written as zeros.  C % 64 == 0, V <= 8. */
GLF_API int glf_views_to_tokens(int B, int C, int V, int T, int src_dtype, const void* const* src,
                        const int64_t* stride_b, const int64_t* stride_c, const int64_t* stride_t, void* out,
                        glf_stream_t stream);

/* ---- data-parallel gradient exchange (replaces nn.DataParallel's reduce onto GPU 0, R/main.py:155) ----------------
 * One kernel over NVLink / NVSwitch peer memory: every rank (one process per GPU) keeps its flat fp32 gradient bucket
 * in a device allocation that the other ranks have opened through CUDA IPC, preceded by a zero-initialised signal pad
 * of glf_p2p_signal_bytes(world) bytes.  glf_p2p_allreduce replaces every rank's bucket, in place, by
 * scale * (sum over ranks), bitwise identical on all ranks; it is CUDA-graph capturable (no host-side state).
 *   setup:  glf_p2p_export(ptr) -> (64-byte handle, offset) on the owner;  glf_p2p_open(handle, offset) on the peers
 *   bufs / sigs: HOST arrays of `world` device pointers (own pointer at index `rank`)
 *   n: floats, multiple of 4, <= glf_p2p_max_floats();  world 2..8;  every rank must call with the same n */
GLF_API size_t glf_p2p_signal_bytes(int world);
GLF_API int64_t glf_p2p_max_floats(void);
GLF_API int glf_p2p_export(const void* ptr, unsigned char handle[64], uint64_t* offset);
GLF_API int glf_p2p_open(const unsigned char handle[64], uint64_t offset, void** out);
GLF_API int glf_p2p_close(void* ptr, uint64_t offset);
GLF_API int glf_p2p_allreduce(void* const* bufs, void* const* sigs, int rank, int world, int64_t n, float scale,
                      glf_stream_t stream);

/* ---- building blocks, exported for unit tests and for callers that fuse differently ------------------------ */

/* D[b] = alpha * A[b] * B[b]^T (+ bias[n]) (+ addend) on tcgen05 tensor cores, bf16 operands, fp32 accumulate.
 *   A: M x K, B: N x K.  a_mn / b_mn = 0: operand stored K-contiguous ([rows, K], leading dim ld);
 *                                     = 1: operand stored MN-contiguous ([K, rows], leading dim ld).
 *   out_kind 0: bf16 store, 1: fp32 store, 2: fp32 atomic add (split_k > 1 requires 2).
 *   colstats (optional): table of partial column sums / sums of squares of the stored values over ALL rows of ALL
 *                        batch entries: zero it, size it [batch * ceil(M/128) * 4][2][N] fp32, and sum its rows (the
 *                        kernel writes one row per (CTA, 32-row quarter) or per (tile, quarter)).
 *   batch strides in elements; strideB = 0 shares B across the batch. */
GLF_API int glf_gemm_bf16(const void* A, const void* B, void* D, int M, int N, int K, int batch, int a_mn, int b_mn,
                  int64_t lda, int64_t ldb, int64_t ldd, int64_t strideA, int64_t strideB, int64_t strideD,
                  const float* bias, float alpha, const void* addend, int64_t ld_add, int64_t stride_add,
                  int out_kind, int split_k, float* colstats, glf_stream_t stream);

/* Same product with the two extras the Gram form of mode='dot' uses (unit tests):
 *   bias_stride : elements between the bias vectors of consecutive batch entries (0 = one shared [N] vector);
 *   rowsum      : optional [batch][M] fp32, rowsum[b][m] = sum_k A[b][m][k] (a side product on the tensor cores:
 *                 A x ones^T into 16 spare TMEM columns); stored, or atomically added when split_k > 1 (zero it). */
GLF_API int glf_gemm_bf16_ex(const void* A, const void* B, void* D, int M, int N, int K, int batch, int a_mn, int b_mn,
                     int64_t lda, int64_t ldb, int64_t ldd, int64_t strideA, int64_t strideB, int64_t strideD,
                     const float* bias, int64_t bias_stride, float alpha, int out_kind, int split_k, float* rowsum,
                     glf_stream_t stream);

/* Token contraction of the Gram form, one CTA per sequence (C = 128 or 256; unit tests, roofline probe):
 *   D[b] = A[b]^T X[b]  with A, X: [B, N, C] bf16 token-major;  D: [B, ldd, ldd] bf16, rows / columns < C written
 *   (ldd >= C, ldd % 8 == 0);  colsum: [B, C] fp32 column sums of A.  A == X gives the Gram matrix S = X^T X. */
GLF_API int glf_gram_contraction(const void* A, const void* X, void* D, float* colsum, int B, int N, int C, int ldd,
                         glf_stream_t stream);

/* The softmax attention of mode='embedded' on its own (unit tests): the functions glf_tpavi_fwd / glf_tpavi_bwd run,
 * with the same head-width dispatch (flash kernels for Ci = 64 and 128, the chunked exact path otherwise).
 *   fwd: Y = softmax(Theta Phi^T) G per sequence, no 1/sqrt(Ci) scale;  lse = logsumexp of each score row (natural log).
 *   bwd: dP3 = [dTheta | dPhi | dG] from dY and the forward's Y and lse;  bias_grad (optional, may be NULL): the 3 Ci
 *        column sums of dP3 over all B * N rows, reduced as glf_tpavi_bwd reduces its bias gradients.
 *   P3: [B, N, 3 Ci] bf16 = [Theta | Phi | G] per token;  Y, dY: [B, N, Ci] bf16;  lse: [B, N] fp32;  dP3 like P3.
 *   B, N > 0;  Ci a positive multiple of 8, <= 2048;  16-byte aligned pointers.
 *   scratch: glf_attention_scratch_bytes(B, N, Ci, backward) bytes, 256-byte aligned (0 = invalid arguments). */
GLF_API size_t glf_attention_scratch_bytes(int B, int N, int Ci, int backward);
GLF_API int glf_attention_fwd(const void* P3, void* Y, float* lse, int B, int N, int Ci, void* scratch, glf_stream_t s);
GLF_API int glf_attention_bwd(const void* P3, const void* Y, const void* dY, const float* lse, void* dP3, float* bias_grad,
                      int B, int N, int Ci, void* scratch, glf_stream_t s);

/* The softmax attention of mode='gaussian' on its own (unit tests): Q = K = X, no projection, no 1/sqrt(C) scale.
 * Flash kernels for (C, Ci) = (64, 64), (128, 64) and (128, 128), the chunked exact path otherwise.
 *   fwd: Y = softmax(X X^T) G per sequence;  lse = logsumexp of each score row (natural log).
 *   bwd: with P = softmax(X X^T), delta = rowsum(dY o Y), dS = P o (dY G^T - delta):
 *        dX = dS X + dS^T X  (each term rounded to bf16, then their fp32 sum rounded once),  dG = P^T dY;
 *        bias_grad (optional, may be NULL): the Ci column sums of dG over all B * N rows (g.bias).
 *   X, dX: [B, N, C] bf16;  G, Y, dY, dG: [B, N, Ci] bf16;  lse: [B, N] fp32.
 *   B, N > 0;  C and Ci positive multiples of 8, at most 2048;  16-byte aligned pointers.
 *   scratch: glf_attention_gaussian_scratch_bytes(B, N, C, Ci, backward) bytes, 256-byte aligned (0 = invalid). */
GLF_API size_t glf_attention_gaussian_scratch_bytes(int B, int N, int C, int Ci, int backward);
GLF_API int glf_attention_gaussian_fwd(const void* X, const void* G, void* Y, float* lse, int B, int N, int C, int Ci,
                               void* scratch, glf_stream_t s);
GLF_API int glf_attention_gaussian_bwd(const void* X, const void* G, const void* Y, const void* dY, const float* lse,
                               void* dX, void* dG, float* bias_grad, int B, int N, int C, int Ci, void* scratch,
                               glf_stream_t s);

/* The two HBM-bound fused epilogues as standalone entry points (unit tests, roofline probes).
 *   fwd: Z = LayerNorm_C(bn_a * U + bn_b + X) * ln_w + ln_b   (ours.py:908-915 after the W_z GEMM); U, X bf16 [rows, C];
 *        Z [rows, C] of z_dtype (bf16, fp16 or fp32); mu, r: per-row LayerNorm mean / rstd (kept for backward).
 *   bwd: dV = d(pre-LayerNorm sum) [rows, C] bf16 from dZ of dz_dtype, and per-CTA partials [nblocks][4][C] of
 *        (d ln_w, d ln_b, d bn_gamma, d bn_beta); *nblocks_out receives the number of partial rows written.
 *        `part` must hold glf_bn_res_ln_bwd_max_blocks() * 4 * C floats. */
GLF_API int glf_bn_res_ln_fwd(int64_t rows, int C, const void* U, const void* X, const float* bn_a, const float* bn_b,
                      const float* ln_w, const float* ln_b, void* Z, int z_dtype, float* mu, float* r, float eps,
                      int accumulate, glf_stream_t stream);
GLF_API int glf_bn_res_ln_bwd(int64_t rows, int C, const void* dZ, int dz_dtype, const void* U, const void* X,
                      const float* bn_a, const float* bn_b, const float* bn_mean, const float* bn_rstd,
                      const float* ln_w, const float* mu, const float* r, void* dV, float* part, int* nblocks_out,
                      glf_stream_t stream);
GLF_API int glf_bn_res_ln_bwd_max_blocks(void);

/* Pair forms (MGFM = index 0, MLFM = index 1) of the two epilogues with explicit operands: every argument that is a
 * pointer-to-pointer is a HOST array of two device pointers.  bf16 activations, C <= 256, 16-byte aligned pointers.
 *   fwd: Z (+)= sum_m LayerNorm_C(bn_a[m] * U[m] + bn_b[m] + X[m]) * ln_w[m] + ln_b[m]
 *   bwd: dV[m] and part[m] ([nblocks][4][C]) for both blocks from ONE read of dZ. */
GLF_API int glf_bn_res_ln_pair_fwd(int64_t rows, int C, const void* const* U, const void* const* X,
                           const float* const* bn_a, const float* const* bn_b, const float* const* ln_w,
                           const float* const* ln_b, void* Z, float* const* mu, float* const* r, float eps,
                           int accumulate, glf_stream_t stream);
GLF_API int glf_bn_res_ln_pair_bwd(int64_t rows, int C, const void* dZ, const void* const* U, const void* const* X,
                           const float* const* bn_a, const float* const* bn_b, const float* const* bn_mean,
                           const float* const* bn_rstd, const float* const* ln_w, const float* const* mu,
                           const float* const* r, void* const* dV, float* const* part, int* nblocks_out,
                           glf_stream_t stream);

/* ---- the cycle-consistency step that consumes the MGFM output (R/main.py:229-235) ---------------------------------
 * glf_spatial_sums: out[b, c] = sum_t x[b, c, t] (fp32) for one view [B, C, h*w] given by element strides — replaces
 *   cyc_feat_out[view].sum(dim=(2, 3)) (R/main.py:229); channels-last views (stride_c == 1, what the fusion path
 *   returns) are read coalesced along C.  dtype: GLF_DTYPE_BF16, GLF_DTYPE_F16 or GLF_DTYPE_F32.
 * glf_cycle_loss: Trainer.seg_cycle (R/main.py:650-717: n_starts = 1, start = the np.random.choice draw, scale = 1)
 *   and Trainer.dense_seg_cycle (R/main.py:719-798: start = 0, step = 1 or chunk_size, n_starts positions, scale =
 *   1 / (target_region - chunk_size - cyc_off + 1), soft_label as there) on the [T, C] fp32 per-frame features.
 *   Writes the scalar loss AND d loss / d feat ([T, C] fp32) in the same call: the loss is a scalar, so the autograd
 *   backward is grad_output * dfeat.  scratch: glf_cycle_loss_scratch_bytes(T, C, n_starts) bytes.  Deterministic. */
GLF_API int glf_spatial_sums(const void* x, int dtype, int B, int C, int T, int64_t stride_b, int64_t stride_c,
                     int64_t stride_t, float* out, glf_stream_t stream);
GLF_API size_t glf_cycle_loss_scratch_bytes(int T, int C, int n_starts);
GLF_API int glf_cycle_loss(const float* feat, int T, int C, int target_region, int cyc_off, int chunk_size,
                   float temperature, int start, int step, int n_starts, int soft_label, float scale, float* loss,
                   float* dfeat, void* scratch, glf_stream_t stream);

/* out[b, s, r] = in[b, r, s] with dtype conversion (NCTHW <-> token-major packing). dtypes: GLF_DTYPE_* (fp16 <-> bf16
 * and fp16 <-> fp32 included). */
GLF_API int glf_transpose(const void* in, void* out, int batch, int R, int S, int in_dtype, int out_dtype,
                  glf_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GLFUSION_H_ */
