/*
 * b2no -- B200-native Fourier-neural-operator hot path (C ABI).
 *
 * Drop-in boundary for the SpectralConv hot path of neuraloperator/pde-policylearning.  The reference is
 * pure Python/PyTorch: it has no FFI of its own, its "operator interface" for this path is the three
 * nn.Module.forward() methods below plus the autograd backward PyTorch derives for them.  Each entry point
 * cites the reference lines it replaces; INTEGRATION.md shows the ctypes stub a reference maintainer adds.
 *
 *   neuralop/models/spectral_convolution.py:303-347   FactorizedSpectralConv.forward      (a1)
 *   neuralop/models/fno_block.py:123-170              FNOBlocks.forward (skip + act)      (a3)
 *   neuralop/models/tfno.py:11-38                     Lifting / Projection                (a3)
 *   neuralop/models/rno.py:60-77,224-228,254-260      SpectralConv2d / FourierLayer2d / RNO_cell (a4,a5)
 *   libs/models/pino_models/basics.py:114-143         SpectralConv3d.forward              (a6)
 *   libs/models/pino_models/pinobserver.py:212-232    pointwise head / tail               (a7)
 *   libs/utilities3.py:323-334                        LpLoss.rel                          (a9)
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; buffers are owned by the caller
 *     (PyTorch); the library allocates only the per-plan twiddle tables.
 *   - `stream` is a cudaStream_t passed as void*; no entry point synchronises the device; all are
 *     CUDA-graph capturable except b2no_plan_create/destroy.
 *   - return value: 0 = ok, negative = bad argument / unsupported shape (B2NO_E_*), positive = cudaError_t.
 *   - real tensors are contiguous fp32 (batch, channel, *grid); spectra are complex64 interleaved
 *     (re,im) laid out (batch*channel, K_1, ..., K_d) over the KEPT modes only.
 *   - there is no CPU fallback: without a CUDA device every compute entry point returns an error.
 */
#ifndef B2NO_H
#define B2NO_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2NO_MAX_DIM 3
#define B2NO_ABI_VERSION 5

enum { B2NO_NORM_BACKWARD = 0, B2NO_NORM_FORWARD = 1, B2NO_NORM_ORTHO = 2 };
enum { B2NO_ACT_NONE = 0, B2NO_ACT_GELU = 1, B2NO_ACT_RELU = 2, B2NO_ACT_SIGMOID = 3, B2NO_ACT_SELU = 4,
       B2NO_ACT_TANH = 5 };
enum { B2NO_E_ARG = -1, B2NO_E_UNSUPPORTED = -2, B2NO_E_NODEVICE = -3 };

/* Geometry of one truncated spectral convolution (mirrors oracle/closed_form.py::SpecGeom).
 *   nin  : physical input grid                      (x.shape[2:])
 *   nfft : forward transform lengths                (== nin, except rno.py:66-67 forces (n, n))
 *   nout : output grid                              (== nfft, except output_scaling_factor,
 *                                                    spectral_convolution.py:339-342)
 *   half : kept modes per dim; dims 0..ndim-2 keep rows [0,h) U [N-h,N), the last dim keeps [0,h)
 */
typedef struct {
  int32_t ndim;
  int32_t nin[B2NO_MAX_DIM];
  int32_t nfft[B2NO_MAX_DIM];
  int32_t nout[B2NO_MAX_DIM];
  int32_t half[B2NO_MAX_DIM];
  int32_t norm;
  /* layout of the kept-mode spectra this plan's transforms write / read and its mixing calls work on:
   *   0  (batch, channel, K_1..K_d)   the default (what a reader of rfftn's output would expect)
   *   1  (K_1..K_d, batch, channel)   mode-major: the per-mode [batch x channel] slab of the mixing GEMMs is contiguous.
   *      2-D plans on the tensor-core transform kernels only (b2no_plan_layout_supported); used by the RNO layer, where
   *      the mixing is real tensor-core work (rno.py:51-58,71-74 at batch 256) */
  int32_t spec_layout;
} b2no_geom;

typedef struct b2no_plan b2no_plan;

/* Complex spectral weights as the reference stores them: one tensor per corner, each (Ci, Co, h_1..h_d)
 * complex64 interleaved -- tltorch ComplexDense (spectral_convolution.py:259-266), rno.py:43-46 real pairs
 * and basics.py:109-112 cfloat Parameters all share this memory layout.  Corner order is canonical:
 * index = sum_j highbit_j * 2^(ndim-2-j) == itertools.product order of spectral_convolution.py:330-337.
 * Strides are in complex elements so incremental_n_modes slices (spectral_convolution.py:276-301) work. */
typedef struct {
  const float* corner[4];
  int64_t stride_i, stride_o;
  int64_t stride_k[B2NO_MAX_DIM];
} b2no_weights;

/* Fused epilogue of the inverse transform:
 *   z = irfft(Yh) + bias[o] + sum_i pw_w[o,i] * pw_x[b,i,.] + sum_i pw2_w[o,i] * pw2_x[b,i,.] + add[b,o,.]
 *   y = act(z) * (mul ? mul[b,o,.] : 1) * (dact_z ? dact'(dact_z[b,o,.]) : 1)
 *       + (gate_z ? (1 - gate_z[b,o,.]) * gate_h[b,o,.] : 0)
 * (fno_block.py:131,142-150; rno.py:224-228,254-259; pinobserver.py:222-226).  pw_w is (Co, Ci) row-major,
 * or (Ci, Co) when pw_transposed (the dx pass of the 1x1 conv).  preact, when non-NULL, receives z.
 * The gate term is the GRU-style state update of rno.py:259, h' = (1 - z) h + z2 hhat, with mul = z2: the candidate
 * state hhat = act(.) never touches HBM.  mul_bstride / gate_bstride (floats between consecutive samples of mul /
 * gate_z; 0 = dense, channels * pixels) let both gates be channel slices of ONE (batch, 2 C, grid) tensor. */
typedef struct {
  const float* bias;
  const float* pw_w;  const float* pw_x;  int32_t pw_ci;  int32_t pw_transposed;
  const float* pw2_w; const float* pw2_x; int32_t pw2_ci; int32_t pw2_transposed;
  const float* add;
  const float* mul;
  float* preact;
  int32_t act;
  /* backward chaining: multiply by the derivative of activation `dact` evaluated at the saved
   * pre-activation dact_z of the PREVIOUS layer, so a layer's dx pass emits gz of the layer below directly */
  const float* dact_z;
  int32_t dact;
  const float* gate_z;
  const float* gate_h;
  int64_t mul_bstride;
  int64_t gate_bstride;
} b2no_epilogue;

int b2no_version(void);
const char* b2no_error_string(int code);
int b2no_device_info(int* sm_count, int* cc_major, int* cc_minor, int64_t* l2_bytes);

/* ---- plans ------------------------------------------------------------------------------------- */
int b2no_plan_create(const b2no_geom* geom, b2no_plan** out);
int b2no_plan_destroy(b2no_plan* plan);
/* 1 when every transform / mixing call of this plan can run with its spec_layout for (batch, channels) tensors */
int b2no_plan_layout_supported(const b2no_plan* plan, int64_t batch, int64_t channels);
/* kept modes per dim (K_j) */
int b2no_plan_kept(const b2no_plan* plan, int32_t kept[B2NO_MAX_DIM]);
/* floats of scratch needed by dft_forward / dft_inverse for a (batch, channels) tensor */
int64_t b2no_plan_workspace_floats(const b2no_plan* plan, int64_t batch, int64_t channels);
/* 1 = use the tcgen05 tensor-core kernels where the shape is eligible (default on sm_100), 0 = CUDA-core kernels
 * only.  Returns the mode now in force.  Both paths are CUDA; neither is a CPU fallback. */
int b2no_set_tensor_core_mode(int on);
/* Tensor-core precision mode (north_star: "<= 1e-5 in fp32, <= 2e-2 when the reduced tensor-core mode is enabled, stated per
 * config"): 0 = fp32-accurate, every product issued three times on tf32 splits (3xTF32; default); 1 = single-pass TF32
 * (one kind::tf32 MMA per product, no hi/lo split work in the issue loop; measured error ~1e-3).  Activations, spectra and
 * weights stay fp32 in HBM in both modes.  Returns the mode now in force. */
int b2no_set_precision(int mode);
/* number of tcgen05 kernel launches issued so far by this process (evidence for tests / bench) */
int64_t b2no_tensor_core_launches(void);

/* ---- truncated transforms ---------------------------------------------------------------------- */
/* which = 0: Xh = s_f * DFT_trunc(x)            x on the nin grid    (rfftn + slicing)
 * which = 1: gYh = adjoint of the inverse       gy on the nout grid  (backward of irfftn) */
int b2no_dft_forward(const b2no_plan* plan, int which, const float* x, float* spec, float* work,
                     int64_t bc, void* stream);
/* which = 0: y  = s_i * Re(IDFT_trunc(Yh)) on the nout grid, fused epilogue       (irfftn + bias ...)
 * which = 1: dx = adjoint of the forward on the nin grid, fused epilogue           (backward of rfftn)
 * spec may be NULL (pure pointwise op: y = act(bias + pw + add)); then `pixels` is the flattened grid. */
int b2no_dft_inverse(const b2no_plan* plan, int which, const float* spec, float* y, float* work,
                     int batch, int channels, int64_t pixels, const b2no_epilogue* epi, void* stream);

/* ---- per-mode channel mixing ------------------------------------------------------------------- */
/* mode 0: Yh[b,o,k]  (+)= sum_i Xh[b,i,k]  * W[i,o,k]          (the einsum, spectral_convolution.py:31-36)
 * mode 1: gXh[b,i,k] (+)= sum_o gYh[b,o,k] * conj(W[i,o,k])    (its input adjoint) */
int b2no_mix(const b2no_plan* plan, int mode, const float* in, const b2no_weights* w, float* out,
             int batch, int ci, int co, int accumulate, void* stream);
/* dW[i,o,k] (+)= sum_b conj(Xh[b,i,k]) * gYh[b,o,k]  written in the reference's corner layout */
int b2no_mix_dw(const b2no_plan* plan, const float* xh, const float* gyh, const b2no_weights* dw,
                int batch, int ci, int co, int accumulate, void* stream);

/* ---- pointwise kernels -------------------------------------------------------------------------- */
/* gz = gy * act'(z)  (elementwise, n floats) */
int b2no_act_bwd(const float* gy, const float* z, float* gz, int64_t n, int act, void* stream);
/* dW[o,i] = sum_{b,p} g[b,o,p] x[b,i,p] ; db[o] = sum_{b,p} g[b,o,p] (db may be NULL).
 * partial: scratch of b2no_pw_wgrad_scratch_floats(ci,co) floats. */
int64_t b2no_pw_wgrad_scratch_floats(int ci, int co);
int b2no_pw_wgrad(const float* g, const float* x, float* dw, float* db, float* partial, int batch, int ci,
                  int co, int64_t pixels, void* stream);
/* The dx pass of a 2-D FNO layer and the weight gradient of its 1x1 skip in one pass over the pixel tiles:
 *   y = b2no_dft_inverse(plan, which, spec, ..., epi)   with epi->pw_x = g (batch, co = epi->pw_ci, pixels)
 *   dw[o,i] = sum_{b,p} g[b,o,p] x[b,i,p] ;  db[o] = sum_{b,p} g[b,o,p] (db may be NULL)      x = wg_x (batch, wg_ci, pixels)
 * -- b2no_dft_inverse followed by b2no_pw_wgrad(g, x), without reading g a second time.  partial: scratch of
 * b2no_pw_wgrad_scratch_floats(wg_ci, co) floats.  Runs on the tensor-core tile kernel only: returns B2NO_E_UNSUPPORTED, having
 * written nothing, when it cannot (not a 2-D plan, no tensor cores, an epilogue with anything but pw_w / pw_x -- bias, act,
 * dact_z, a second 1x1 operand --, co > 64, wg_ci > 112, pixels % 128 != 0, misaligned pointers, shared memory too small);
 * the caller then makes the two calls. */
int b2no_dft_inverse_wgrad(const b2no_plan* plan, int which, const float* spec, float* y, float* work, int batch, int channels,
                           int64_t pixels, const b2no_epilogue* epi, const float* wg_x, int wg_ci, float* dw, float* db,
                           float* partial, void* stream);
/* fused projection head (tfno.py:34-38; pinobserver.py:230-232 after folding MultiplicativeNet):
 *   out[b,p] = b2 + sum_j w2[j] * gelu( b1[(b),j] + sum_i w1[j,i] x[b,i,p] )      (out_channels == 1)
 * b1 is (hidden) or, when b1_per_sample, (batch, hidden). */
int b2no_mlp_head_fwd(const float* x, const float* w1, const float* b1, const float* w2, const float* b2,
                      float* out, int batch, int ci, int hidden, int64_t pixels, int b1_per_sample,
                      int act, void* stream);
/* input-gradient half of the backward of the fused head (hidden activations recomputed on the tensor cores):
 *   f[b,j,p] = g[b,p] w2[j] act'(z1[b,j,p]);  gx[b,i,p] = sum_j w1[j,i] f[b,j,p] (* dact'(dact_z) when given);
 *   dw2[j] = sum_{b,p} g[b,p] act(z1[b,j,p]);  gz (optional, (batch, hidden, pixels)) receives f for b2no_pw_wgrad.
 * partial: b2no_mlp_head_bwd_scratch_floats(hidden) floats.  Returns B2NO_E_UNSUPPORTED when the shape has no
 * tensor-core kernel (the caller then composes the pointwise entry points). */
int64_t b2no_mlp_head_bwd_scratch_floats(int hidden);
int b2no_mlp_head_bwd_supported(int ci, int hidden, int64_t pixels);
int b2no_mlp_head_bwd(const float* x, const float* w1, const float* b1, const float* w2, const float* g, float* gx,
                      float* gz, float* dw2, float* partial, int batch, int ci, int hidden, int64_t pixels,
                      int b1_per_sample, int act, const float* dact_z, int dact, void* stream);
/* WHOLE backward of the fused head in one kernel (same reference lines; replaces b2no_mlp_head_bwd + b2no_pw_wgrad on the
 * hidden-channel gradient): f is recomputed on the tensor cores and never written to memory.
 *   gx[b,i,p] as above;  grads = [ dW1 (hidden x ci) | db1 (hidden) | dw2 (hidden) | db2 (1) ] contiguous floats:
 *   dW1[j,i] = sum_{b,p} f[b,j,p] x[b,i,p];  db1[j] = sum_{b,p} f[b,j,p];  dw2[j] = sum_{b,p} g[b,p] act(z1[b,j,p]);
 *   db2 = sum_{b,p} g[b,p].
 * b1 is (hidden) (a per-sample bias keeps the two-kernel path).  partial: b2no_mlp_head_bwd_fused_scratch_floats(ci, hidden)
 * floats.  Shapes: ci <= 32, hidden <= 256, pixels % 128 == 0 (b2no_mlp_head_bwd_fused_supported); otherwise
 * B2NO_E_UNSUPPORTED. */
int64_t b2no_mlp_head_bwd_fused_scratch_floats(int ci, int hidden);
int b2no_mlp_head_bwd_fused_supported(int ci, int hidden, int64_t pixels);
int b2no_mlp_head_bwd_fused(const float* x, const float* w1, const float* b1, const float* w2, const float* g, float* gx,
                            float* grads, float* partial, int batch, int ci, int hidden, int64_t pixels, int act,
                            const float* dact_z, int dact, void* stream);
/* Fused head with out_channels = O = 2..4 (pinobserver.py:230-232 via PlanePredHead, :257-273, whose tail emits
 * plane_num * out_dim channels; tfno.py:34-38 Projection with out_channels > 1):
 *   out[b,o,p] = b2[o] + sum_j w2[o,j] * act( b1[(b),j] + sum_i w1[j,i] x[b,i,p] )
 * w2 is (O, hidden) row-major, b2 (O) or NULL, out (batch, O, pixels); the hidden tensor is never written.  Tensor cores
 * only: returns B2NO_E_UNSUPPORTED, having written nothing, when O is outside 2..4, pixels % 128 != 0, ci > 64,
 * hidden > 512, x is not 16-byte aligned, the device has no tensor-core kernels or shared / tensor memory is too small. */
int b2no_mlp_head_fwd_multi(const float* x, const float* w1, const float* b1, const float* w2, const float* b2, float* out,
                            int batch, int ci, int hidden, int out_channels, int64_t pixels, int b1_per_sample, int act,
                            void* stream);
/* Input-gradient half of its backward, the O-output form of b2no_mlp_head_bwd (same reference lines):
 *   f[b,j,p] = act'(z1[b,j,p]) sum_o g[b,o,p] w2[o,j];  gx[b,i,p] = sum_j w1[j,i] f[b,j,p] (* dact'(dact_z) when given);
 *   dw2[o,j] = sum_{b,p} g[b,o,p] act(z1[b,j,p]) ((O, hidden));  gz (optional, (batch, hidden, pixels)) receives f for
 *   b2no_pw_wgrad (dW1, db1).  g is (batch, O, pixels).  partial: b2no_mlp_head_bwd_multi_scratch_floats(hidden, O) floats.
 * Returns B2NO_E_UNSUPPORTED, having written nothing, where b2no_mlp_head_bwd_multi_supported is 0 (same limits as the
 * forward, and the shared-memory budget of the backward: e.g. ci = 64 with hidden = 256 does not fit). */
int b2no_mlp_head_bwd_multi_supported(int ci, int hidden, int out_channels, int64_t pixels);
int64_t b2no_mlp_head_bwd_multi_scratch_floats(int hidden, int out_channels);
int b2no_mlp_head_bwd_multi(const float* x, const float* w1, const float* b1, const float* w2, const float* g, float* gx,
                            float* gz, float* dw2, float* partial, int batch, int ci, int hidden, int out_channels,
                            int64_t pixels, int b1_per_sample, int act, const float* dact_z, int dact, void* stream);
/* RNO gate (rno.py:259): h_next = (1 - z) * h + z2 * hhat, and its backward */
int b2no_rno_gate_fwd(const float* z, const float* z2, const float* hhat, const float* h, float* out,
                      int64_t n, void* stream);
int b2no_rno_gate_bwd(const float* g, const float* z, const float* z2, const float* hhat, const float* h,
                      float* gz, float* gz2, float* ghhat, float* gh, int64_t n, void* stream);
/* Backward of the fused RNO cell update (rno.py:254-259), emitting the PRE-activation gradients of all gates at once:
 *   h' = (1 - z) h + z2 selu(ah),  z = sigmoid(az), z2 = sigmoid(az2)   (zz2 = [z | z2] post-sigmoid, (batch, 2C, pixels))
 *   g_zz2[:, :C] = -g h z (1 - z);  g_zz2[:, C:] = g selu(ah) z2 (1 - z2);  g_ah = g z2 selu'(ah);  g_h = g (1 - z)
 * and of the reset gate r = sigmoid(ar) inside f6(r * h):
 *   g_ar = g_rh h r (1 - r);  g_h += g_rh r
 * n = batch, c = channels, p = pixels per channel; every tensor is dense (batch, channels, pixels). */
int b2no_rno_cell_bwd(const float* g, const float* h, const float* zz2, const float* ah, float* g_zz2, float* g_ah,
                      float* g_h, int batch, int c, int64_t p, void* stream);
int b2no_rno_reset_bwd(const float* g_rh, const float* h, const float* ar, float* g_ar, float* g_h, int64_t n,
                       void* stream);
/* LpLoss.rel, p=2 (utilities3.py:323-334): per-sample sums -> sums[b] = (||x-y||^2, ||y||^2) */
int b2no_rel_l2_sums(const float* x, const float* y, float* sums, int batch, int64_t n_per_sample, void* stream);
/* dx = coef[b] * (x - y)  with coef[b] precomputed by the host from sums (and the upstream gradient) */
int b2no_rel_l2_bwd(const float* x, const float* y, const float* coef, float* dx, int batch,
                    int64_t n_per_sample, void* stream);
/* Device-side tail of LpLoss.rel (utilities3.py:331-334): loss = sum_b (size_average: mean_b) of sqrt(sums[b][0]) /
 * sqrt(sums[b][1]); coef[b] (optional) = scale / (||x_b - y_b|| ||y_b||), the factor of the backward. */
int b2no_rel_l2_finish(const float* sums, float* loss, float* coef, int batch, int size_average, void* stream);
/* dx = g[0] * coef[b] * (x - y): backward of LpLoss.rel with the upstream scalar gradient g read on the device */
int b2no_rel_l2_bwd_g(const float* x, const float* y, const float* coef, const float* g, float* dx, int batch,
                      int64_t n_per_sample, void* stream);

/* ---- PINO PDE-residual loss (SURVEY 8a row a8, 8f rank 3) ------------------------------------------ */
/* Fused Channelflow_PINO_loss (libs/envs/diff_control_env.py:44-60) with FDM_NS_vorticity (:5-41) inside: one CTA per
 * (sample, time slice) does the spectral derivatives as mode-restricted DFT contractions in shared memory, the products,
 * the central difference in t and the warp-shuffle partial sums of both relative-L2 losses.
 *   w (B, N, N, T) model output, t fastest; u0 (B, N, N); forcing (N, N); nu (B,) = 1 / Re; N % 4 == 0, 8 <= N <= 64.
 *   du_p (B, T, N, N): residual planes 1 .. T-2 (plane-contiguous); fields (4, B, T, N, N): ux, wx, uy, wy for the backward;
 *   partial (B, T, 4) scratch; loss[0] = loss_ic, loss[1] = loss_f; coef (B, 2) = the factors of the backward.
 * bwd: dw (B, N, N, T) = gup[0] d loss_ic / dw + gup[1] d loss_f / dw (gup: 2 floats on the device). */
int64_t b2no_pino_residual_scratch_floats(int B, int N, int T, int which);
int b2no_pino_residual_fwd(const float* w, const float* u0, const float* forcing, const float* nu, float t_interval,
                           float* du_p, float* fields, float* partial, float* loss, float* coef, int B, int N, int T,
                           void* stream);
int b2no_pino_residual_bwd(const float* w, const float* u0, const float* forcing, const float* nu, float t_interval,
                           const float* du_p, const float* fields, const float* coef, const float* gup, float* dw,
                           int B, int N, int T, void* stream);

/* ---- optimizer (SURVEY 8f rank 2) ---------------------------------------------------------------- */
/* One fused Adam update over a flat fp32 buffer (complex parameters as their (re, im) view), torch.optim.Adam
 * semantics as the reference configures it (run_pde_observers.py:134, train_pino.py:205): L2 weight decay,
 * bias correction.  grad_scale multiplies the gradient first (1/world_size after a sum all-reduce).
 * step_counter is a DEVICE int incremented by the call, so a captured CUDA graph replays correctly. */
int b2no_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, int* step_counter,
                   float lr, float beta1, float beta2, float eps, float weight_decay, float grad_scale, void* stream);
/* number of kernels this library has launched so far in this process (host-side counter; kernels replayed from a
 * captured CUDA graph are not seen by it) */
int64_t b2no_kernel_launches(void);

/* flat[offsets[s] .. offsets[s+1]) = src_ptrs[s][0 .. counts[s]) (zero fill beyond counts[s] or when src_ptrs[s] is
 * null): the per-parameter gradients autograd produced, gathered into the flat bucket the all-reduce and
 * b2no_adam_step work on.  src_ptrs (nseg device pointers), offsets (nseg + 1) and counts (nseg) are DEVICE arrays.
 * Replaces the per-parameter `p.grad += g` of run_pde_observers.py:192 (loss.backward()). */
int b2no_gather_segments(float* flat, const void* src_ptrs, const int64_t* offsets, const int64_t* counts, int nseg,
                         void* stream);

/* ---- measurement ---------------------------------------------------------------------------------- */
/* Dense tcgen05.mma issue-rate probe for the roofline denominators (SURVEY.md 8d: "measure a kind::tf32 GEMM on the box"):
 * every SM issues n_mma back-to-back M=128, N=256 MMAs from resident shared-memory operands.  kind 0 = kind::tf32,
 * 1 = kind::f16 (bf16 operands).  *flops receives the operation count of the launch; the caller times it with CUDA events. */
int b2no_tc_peak_probe(int kind, int n_mma, double* flops, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B2NO_H */
