/*
 * bayesrul_b200 -- C ABI of the B200-native Monte-Carlo variational-BNN hot path.
 *
 * This is the drop-in boundary for ONE path of lbasora/bayesrul: the weight-sampled forward,
 * ELBO backward and S-sample predictive-moment reduction of its N-CMAPSS regressors.
 * The reference has no FFI (it is pure Python on top of TyXe/Pyro/torch, SURVEY.md F1/F2), so each
 * entry point below names the Python call sequence it replaces (file:line under
 * /root/reference/bayesrul unless prefixed); INTEGRATION.md shows the ctypes stubs a bayesrul
 * maintainer would add.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer to contiguous fp32 unless stated otherwise; tensors are
 *    allocated and owned by the caller (PyTorch caching allocator on the Python side);
 *  - `stream` is a cudaStream_t passed as void*; no entry point synchronises the host;
 *  - every function returns BRL_OK (0) or a negative error code; brl_last_error() gives the text;
 *  - variational parameters are two flat [P] buffers (mu, sigma) in named_parameters() order
 *    (weight then bias per layer) -- brl_net_site() gives per-site offsets so the host can expose
 *    `{site}.loc` / `{site}.scale` views compatible with pyro.get_param_store() (bayesian.py:255-264);
 *  - noise is counter-based Philox4x32-10 keyed by (seed, kind, layer, MC sample, global window,
 *    element), or injected tensors (brl_noise), see csrc/brl_philox.cuh.
 */
#ifndef BAYESRUL_B200_H
#define BAYESRUL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BRL_OK 0
#define BRL_ERR_INVALID (-1)   /* bad argument (shape, enum, NULL) */
#define BRL_ERR_CUDA (-2)      /* CUDA runtime error */
#define BRL_ERR_WORKSPACE (-3) /* workspace too small */
#define BRL_ERR_UNSUPPORTED (-4)

/* nets: models/nets/inception.py:142-217, conv.py:14-79, linear.py:10-72 */
#define BRL_NET_INCEPTION 0
#define BRL_NET_CONV 1
#define BRL_NET_LINEAR 2

/* per-layer rule */
#define BRL_MODE_DET 0     /* plain weights `theta` shared by all S passes (HNN, MC-dropout) */
#define BRL_MODE_WS 1      /* one full weight draw per MC sample: `wsamp` [S,P] (tyxe VariationalBNN.predict) */
#define BRL_MODE_LRT 2     /* tyxe.poutine.local_reparameterization (bayesian.py:66-67) */
#define BRL_MODE_FLIPOUT 3 /* tyxe.poutine.flipout (bayesian.py:68-69) */

#define BRL_GUIDE_NORMAL 0 /* tyxe.guides.AutoNormal (bayesian.py:79-80) */
#define BRL_GUIDE_RADIAL 1 /* AutoRadial / RadialNormal.rsample (guides/radial.py:31-41) */

/* arithmetic back-ends of the forward pass */
#define BRL_ENGINE_SIMT_FP32 0 /* fp32 FFMA implicit-GEMM kernels: the parity engine (rtol 1e-3 vs oracle) */
#define BRL_ENGINE_TC_FP16 1   /* tcgen05 / TMEM kernels, fp16 operands (10-bit mantissa) + fp32 accumulate (every net; dropout: Inception only) */

/* contraction back-ends of the per-layer kernels (every net, every mode, forward + backward) */
#define BRL_GEMM_SIMT_FP32 0 /* fp32 FFMA implicit GEMMs: the parity back-end (rtol 1e-3 vs oracle) */
#define BRL_GEMM_TC_TF32 7   /* tcgen05 kind::tf32 dual GEMMs, fp32 accumulation in TMEM (stated bound 5e-3 vs fp32);
                              * bit mask: 1 forward, 2 input-gradient, 4 weight-gradient kernels (partial masks: debugging) */

#define BRL_GEMM_TC_FUSED 8  /* Inception: brl_elbo_step (LRT / Flipout / weight sampling) and brl_hnn_step (dropout masks in the epilogues)
                              * run the ten conv layers and the fc layer as LEVEL-FUSED tcgen05 kernels (one CTA
                              * per layer per 4-window tile; operands are bulk-copied activation / weight images, taps are
                              * descriptor shifts, the backward contractions read the same images through MN-major descriptors;
                              * fp16 / bf16 operands, fp32 accumulation: outputs 1e-2, loss 5e-3, gradient cosine > 0.999).
                              * Linear: the same two steps run the four hidden layers as tcgen05 GEMMs over 128-window tiles;
                              * Conv-D3: they run the three convs as tcgen05 GEMMs over (window, output position) rows of
                              * im2col images.  Both with the same operand precision and bound, when the workspace holds their
                              * images (brl_workspace_bytes(B, S, 1) includes them), else the per-layer kernels */

#define BRL_MAX_LAYERS 16

typedef struct brl_ctx brl_ctx;

/* Noise specification.  NULL injected pointers => in-kernel Philox keyed by `seed`.
 * Injected layouts (S = MC samples / particles of this call, B = windows of this call):
 *   weight_eps [S,P]        standard normals for the guide draw                      (A7)
 *   radial_r   [S,n_sites]  radial distance, one scalar per site per draw            (A8)
 *   lrt_eps[l]  [S,B,out_elems(l)]  eps of layer l's output                          (A5)
 *   flip_in[l]  [S,B,Cin(l)], flip_out[l] [S,B,Cout(l)]  +-1 sign tensors            (A6)
 *   drop_mask[l] [S,B,out_elems(l)] 0/1 keep masks of the dropout site after layer l (A4)   */
typedef struct brl_noise {
  uint64_t seed;
  int64_t sample0; /* global index of the first MC sample / particle of this call */
  int64_t window0; /* global index of the first window of this call (multi-GPU sharding) */
  const float* weight_eps;
  const float* radial_r;
  const float* lrt_eps[BRL_MAX_LAYERS];
  const float* flip_in[BRL_MAX_LAYERS];
  const float* flip_out[BRL_MAX_LAYERS];
  const float* drop_mask[BRL_MAX_LAYERS];
} brl_noise;

/* ---- library / static net description ------------------------------------------------ */
int brl_version(void);
const char* brl_last_error(void);
/* number of CUDA kernels this library has launched since it was loaded (bench.py gpu_launches) */
int64_t brl_launch_count(void);
int brl_net_num_params(int net);
int brl_net_num_layers(int net);
int brl_net_num_sites(int net);
/* site j of named_parameters(): flat offset, rank and shape (nets/*.py parameter order) */
int brl_net_site(int net, int site, int64_t* offset, int* ndim, int64_t shape[4]);
/* layer l: Cout, C_in seen by flipout, elements of its per-window output, dropout factor
 * (fraction of p applied at the site after this layer: inception.py:48-52,119-123,204-206) */
int brl_net_layer(int net, int layer, int* cout, int* cin, int* out_elems, float* dropout_factor);
/* algorithmic GEMM FLOPs of one forward pass of one window (SURVEY 8(d)) */
int64_t brl_net_flops_fwd(int net);

/* ---- context ------------------------------------------------------------------------- */
int brl_create(brl_ctx** ctx, int net, int device);
int brl_destroy(brl_ctx* ctx);
/* bytes of scratch needed by the calls below for B windows x S concurrently-resident samples;
 * train == 1 adds the saved activations / gradient buffers of brl_elbo_step / brl_hnn_step (with S >= 2: a second set, so
 * that brl_elbo_step runs two particles side by side on two stream lanes),
 * train == 2 the sign tensors brl_forward generates in BRL_MODE_FLIPOUT when none are injected,
 * train == 3 the buffers of brl_hnn_step_ensemble over S = M members (all of them in one chain of launches where it can),
 * train == 4 the buffers of brl_elbo_step_ensemble over S = M members (the same, one particle lane of M members),
 * train == 5 the buffers of brl_elbo_train_steps over S = M members (its own, then those of code 4, or of code 1 with S = 2 at M = 1),
 * train == 6 the buffers of brl_hnn_train_steps over S = M members (its own, then those of code 3, or of code 1 at M = 1),
 * train == 7 the buffers of brl_elbo_val_steps with S predictive samples on `engine` (its own for up to 8 particles, then the larger
 *            of code 1 at S = 2 with engine 0 and the predictive's [S,P] draws and forward workspace) */
/* 1 when `engine` can run this net's forward on this build, else 0 */
int brl_engine_available(const brl_ctx* ctx, int engine);
int64_t brl_workspace_bytes(const brl_ctx* ctx, int64_t B, int64_t S, int train, int engine);
/* tensor-core engine health: 0 = ok, > 0 = code of the first mbarrier wait that timed out inside a
 * tcgen05 kernel (waits are bounded so a protocol bug ends the kernel instead of hanging the GPU),
 * < 0 = engine unavailable.  Synchronises the device. */
int brl_tc_status(const brl_ctx* ctx);
/* Selects how the per-layer kernels of brl_forward (BRL_ENGINE_SIMT_FP32), brl_elbo_step and brl_hnn_step contract:
 * fp32 FFMA (default) or tcgen05 TF32.  Operators, noise, epilogues and results' layout are identical. */
int brl_set_gemm_backend(brl_ctx* ctx, int backend);
/* health of the TF32 per-layer kernels: 0 = ok, > 0 = code of the first bounded mbarrier wait that timed out. Synchronises. */
int brl_gemm_status(void);
/* Measurement hooks of the tensor-core engine (bench.py roofline; no reference counterpart).
 * brl_tc_timing(ctx, 1) starts bracketing every launch of the two tcgen05 kernels with CUDA events on the
 * launching stream; brl_tc_timing_read synchronises those events and returns, for [0] tc_conv_kernel and
 * [1] tc_fc_kernel, the summed kernel milliseconds and the number of launches since the last enable / read;
 * brl_tc_timing(ctx, 0) stops. */
int brl_tc_timing(brl_ctx* ctx, int enable);
int brl_tc_timing_read(brl_ctx* ctx, double kernel_ms[2], int64_t launches[2]);
/* Debug: device buffer (int64[>= 16*128], or NULL to switch off) into which CTA 0 of tc_conv_kernel writes
 * clock64() time stamps of its issuer / epilogue warps for its first 16 work items. */
int brl_tc_trace(brl_ctx* ctx, int64_t* device_buf);
/* Debug: device buffer int64[6 * 4 * 16] (or NULL to switch off) into which CTA (0, layer) of the three forward and the three
 * backward level launches of the BRL_GEMM_TC_FUSED training kernels write clock64() stamps of their phases
 * (start, copies issued, copies landed, operands built, MMAs done, epilogue done, ...). */
int brl_tt_trace(brl_ctx* ctx, int64_t* device_buf);

/* ---- guide: weight sampler (replaces AutoNormal.forward / AutoRadial.forward,
 *      guides/radial.py:31-41,124-144; 24 pyro.sample sites per draw) ------------------- */
int brl_sample_weights(brl_ctx* ctx, const float* mu, const float* sigma, int guide, int64_t S,
                       const brl_noise* noise, float* w_out /*[S,P]*/, float* delta_out /*[S,P] or NULL*/,
                       void* workspace, size_t workspace_bytes, void* stream);

/* ---- forward of S passes over B windows (replaces net.forward under the TyXe messengers,
 *      inception.py:211-215 + tyxe reparameterization_messengers; SURVEY 3.5) -------------
 * x [B,30,18]; theta [P] (DET: weights, LRT/FLIPOUT: mu); sigma [P] (LRT); wsamp [S,P] (WS, FLIPOUT);
 * out [S,B,2] = (loc, scale) after softplus + Threshold(1e-9). */
int brl_forward(brl_ctx* ctx, const float* x, int64_t B, int64_t S, int mode, const float* theta,
                const float* sigma, const float* wsamp, float p_dropout, const brl_noise* noise,
                float* out, int engine, void* workspace, size_t workspace_bytes, void* stream);

/* ---- S-sample predictive moments (replaces bnn.predict(aggregate=False) + bayesian.py:242-249,
 *      and HNN.mc_sampling + frequentist.py:141-146).  guide < 0 => MC-dropout/deterministic with
 *      weights `mu`.  Samples are generated and consumed in chunks that fit the workspace; the
 *      [S,B,2] tensor is never materialised.  Outputs [B] each. */
int brl_predict_moments(brl_ctx* ctx, const float* x, int64_t B, int64_t S, int guide, const float* mu,
                        const float* sigma, float p_dropout, const brl_noise* noise, float* pred,
                        float* std, float* ep_var, float* al_var, int engine, void* workspace,
                        size_t workspace_bytes, void* stream);

/* ---- M models' S-sample predictive moments over ONE batch of windows in one call (the seeds of a BNN experiment or the members
 *      of a deep ensemble at test / predict / validation time).
 *      Member m is brl_predict_moments(x, B, S, guide, mu + m*P, sigma + m*P, p_dropout, noise with sample0 + m*S, ...):
 *      guide >= 0: M variational posteriors (the seeds of a BNN experiment), weight sampling;
 *      guide < 0 : M weight vectors (deep-ensemble members), MC-dropout when p_dropout > 0.
 *      Injected noise is member-major, sample-minor: weight_eps [M*S,P], radial_r [M*S,n_sites], drop_mask[l] [M*S,B,out_elems(l)].
 *      out [4][M][B] = (pred, std, ep_var, al_var), so out + 0 and out + M*B are the [M,B] inputs of brl_mixture_moments.
 *      Each member's results are bit-identical to its single call on the same engine.  On BRL_ENGINE_TC_FP16 the M*S draws form
 *      one sample axis j = m*S + s, cut into chunks that fit the workspace; per chunk the members share one sampler, one pack,
 *      the engine's and one moment-update launch, so a call whose M*S draws fit one chunk issues as many launches as one
 *      member's call.  Elsewhere (SIMT engine; MC-dropout on the Linear and Conv-D3 nets, which the tensor-core engine refuses)
 *      the members run one after another on brl_predict_moments.  Workspace: at least brl_workspace_bytes(B, 1, 0, engine) plus
 *      the [M,4,B] float Welford state (rounded up to 256 bytes); more workspace gives larger chunks.  Less returns
 *      BRL_ERR_WORKSPACE. */
int brl_predict_moments_ensemble(brl_ctx* ctx, const float* x /*[B,30,18]*/, int64_t M, int64_t B, int64_t S, int guide,
                                 const float* mu /*[M,P]*/, const float* sigma /*[M,P] or NULL*/, float p_dropout,
                                 const brl_noise* noise, float* out /*[4,M,B]*/, int engine, void* workspace,
                                 size_t workspace_bytes, void* stream);

/* ---- the same with HOST buffers (replaces predict_step as a whole, bayesian.py:231-250: `x.to(device)`, bnn.predict,
 *      the moments and the five `.cpu()` reads).  x_host [B,30,18] and out_host [4,B] = (pred, std, ep_var, al_var) are HOST
 *      pointers (pinned memory makes the copies asynchronous).  On the fused engine the batch travels in window chunks on a
 *      private copy stream while the previous chunk is computed; the fp16 weight images of all S samples are packed once
 *      and shared by the chunks, so only the first chunk's copy is exposed.  Results equal brl_predict_moments (a weight
 *      draw has no window index; per-window noise is keyed by the global window index).  Nothing synchronises the host:
 *      out_host is valid once `stream` has been synchronised.  Workspace: brl_workspace_bytes_host. */
int64_t brl_workspace_bytes_host(const brl_ctx* ctx, int64_t B, int64_t S, int engine);
int brl_predict_moments_host(brl_ctx* ctx, const float* x_host, int64_t B, int64_t S, int guide, const float* mu,
                             const float* sigma, float p_dropout, const brl_noise* noise, float* out_host /*[4,B]*/,
                             int engine, void* workspace, size_t workspace_bytes, void* stream);

/* moment reduction of an explicit [S,B,2] tensor (bayesian.py:212-215) */
int brl_moments(const float* out, int64_t S, int64_t B, float* pred, float* std, float* ep_var,
                float* al_var, void* stream);
/* tyxe HeteroskedasticGaussian.aggregate_predictions, positive_scale=False (bayesian.py:149-153) */
int brl_aggregate_predictions(const float* out, int64_t S, int64_t B, float* agg /*[B,2]*/, void* stream);

/* ---- one ELBO step: forward + backward (replaces svi.step: bayesian.py:111-132,147) -----
 * loss = mean_particles c*[(N/B)*NLL_sum + KL], c = 1/(N*win_length*n_features).
 * guide RADIAL uses the sampled KL of Trace_ELBO (bayesian.py:105-109) and mode WS.
 * scalars (device, double[4]) = {loss, nll_sum (mean over particles), kl (unscaled), mse(loc,y)}.
 * grad_mu/grad_sigma/grad_log_sigma [P] (any may be NULL when compute_grads == 0).
 * out [particles,B,2]. */
int brl_elbo_step(brl_ctx* ctx, const float* x, const float* y, int64_t B, const float* mu,
                  const float* sigma, int mode, int guide, int particles, float prior_loc,
                  float prior_scale, int64_t dataset_size, const brl_noise* noise, int compute_grads,
                  double* scalars, float* grad_mu, float* grad_sigma, float* grad_log_sigma, float* out,
                  void* workspace, size_t workspace_bytes, void* stream);

/* ---- M independent variational posteriors (the seeds of a BNN experiment) in ONE ELBO step.
 *      Member m is brl_elbo_step(x + m*B*540, y + m*B, B, mu + m*P, sigma + m*P, mode, guide, particles, prior_loc,
 *      prior_scale, dataset_size, noise with sample0 + m*particles, ...): mode, guide, particles, prior, dataset size and seed
 *      are shared; particle pt of member m draws with MC-sample index sample0 + m*particles + pt.  Injected noise is
 *      member-major, particle-minor (member m's tensors are rows [m*particles, (m+1)*particles)): weight_eps [M*particles,P],
 *      radial_r [M*particles,n_sites], lrt_eps[l] [M*particles,B,out_elems(l)], flip_in[l] / flip_out[l] [M*particles,B,C].
 *      Graph-replayed under the same conditions as brl_elbo_step.  brl_clipped_adam_vi over n = M*P is elementwise: M
 *      independent optimisers.
 *      Where brl_elbo_step runs the fused Inception kernels (BRL_GEMM_TC_FUSED; LRT, Flipout or weight sampling; B <= 4736)
 *      and the workspace holds brl_workspace_bytes(B, M, 4), the M members share every launch: one weight-sampler and one
 *      sign-generator launch per particle for all members, the fused forward / fc / tail / backward / reduction kernels with
 *      member = blockIdx.z, the finalisation over M*P with per-member KL, and one scalars launch; the particles run one after
 *      another.  Otherwise (simt / tc back-ends, Linear and Conv-D3 nets, B > 4736, a workspace that holds one member only,
 *      Flipout with several particles and only some of the sign tensors injected) the members run one after another on
 *      brl_elbo_step, with the same results.  A workspace below the single-member size returns BRL_ERR_WORKSPACE. */
int brl_elbo_step_ensemble(brl_ctx* ctx, const float* x /*[M,B,30,18]*/, const float* y /*[M,B]*/, int64_t M, int64_t B,
                           const float* mu /*[M,P]*/, const float* sigma /*[M,P]*/, int mode, int guide, int particles,
                           float prior_loc, float prior_scale, int64_t dataset_size, const brl_noise* noise, int compute_grads,
                           double* scalars /*[M,4] = {loss, nll_sum, kl, mse}*/, float* grad_mu /*[M,P]*/,
                           float* grad_sigma /*[M,P]*/, float* grad_log_sigma /*[M,P] or NULL*/,
                           float* out /*[M,particles,B,2]*/, void* workspace, size_t workspace_bytes, void* stream);

/* brl_elbo_step replays a CUDA graph of the step when the noise is native Philox (no injected tensor): the first call with
 * a given configuration (sizes, mode, parameter / workspace pointers) runs eagerly, the second captures it, later calls
 * replay it with the per-step Philox key {seed, sample0, window0} rewritten in device memory; x, y and the results go
 * through staging buffers inside the workspace, so the caller's tensors may change from step to step.  Results are
 * identical to the eager path.  enable = 0 switches the replay off (also: environment BRL_NO_GRAPH=1). */
int brl_set_step_graph(brl_ctx* ctx, int enable);

/* ---- heteroscedastic NN step (replaces HNN.step + backward: frequentist.py:39-48) ------
 * loss = F.gaussian_nll_loss(loc, y, scale^2); scalars (device double[2]) = {loss, mse}.
 * Replayed as a CUDA graph under the same conditions as brl_elbo_step (native dropout masks or none; key = sizes,
 * p_dropout, theta / workspace pointers). */
int brl_hnn_step(brl_ctx* ctx, const float* x, const float* y, int64_t B, const float* theta,
                 float p_dropout, const brl_noise* noise, int compute_grads, double* scalars,
                 float* grad_theta, float* out /*[B,2]*/, void* workspace, size_t workspace_bytes,
                 void* stream);

/* ---- M independent heteroscedastic NNs (the members of a deep ensemble, models/deepens.py) in ONE step.
 *      Member m is brl_hnn_step(x + m*B*540, y + m*B, B, theta + m*P, p_dropout, noise with sample0 + m, ...):
 *      same loss (F.gaussian_nll_loss over the member's B windows), same dropout keys with MC-sample index sample0 + m,
 *      injected drop_mask[l] laid out [M,B,out_elems(l)].  Graph-replayed under the same conditions as brl_hnn_step.
 *      Where brl_hnn_step runs the fused Inception kernels (BRL_GEMM_TC_FUSED, B <= 4736) and the workspace holds
 *      brl_workspace_bytes(B, M, 3), the M members share every launch (member = blockIdx.z); otherwise they run one after
 *      another on the single-member step, with the same results.  A workspace below the single-member size returns
 *      BRL_ERR_WORKSPACE. */
int brl_hnn_step_ensemble(brl_ctx* ctx, const float* x /*[M,B,30,18]*/, const float* y /*[M,B]*/, int64_t M, int64_t B,
                          const float* theta /*[M,P]*/, float p_dropout, const brl_noise* noise, int compute_grads,
                          double* scalars /*[M,2] = {loss, mse}*/, float* grad_theta /*[M,P]*/, float* out /*[M,B,2]*/,
                          void* workspace, size_t workspace_bytes, void* stream);

/* ---- K consecutive training steps in ONE call, over a device-resident dataset (replaces the epoch loop of Lightning's fit:
 *      DataLoader collate + copy, svi.step / HNN.step, the optimiser, the logged step metrics and their .item() reads, per batch).
 *      X [N,30,18] (16-byte aligned) and Y [N] are the training split; idx [K,M,B] (int64, device) holds the windows of member m's
 *      minibatch at step k.  Step k does exactly:
 *        1. brl_elbo_step_ensemble (brl_elbo_step at M = 1) on X[idx[k]], Y[idx[k]] with the Philox key
 *           {seed + 0x9E3779B97F4A7C15 (k + 1) mod 2^64, sample0, window0} (the key sequence of the reference's per-step seeds);
 *           brl_hnn_train_steps: brl_hnn_step_ensemble (brl_hnn_step at M = 1);
 *        2. brl_clipped_adam_vi (ELBO: loc / log_scale / scale with their moments) or brl_clipped_adam (HNN: theta) over M*P
 *           elements at Adam step step0 + k + 1, with the step size brl_clipped_adam computes;
 *        3. brl_step_metrics_ensemble of particle 0's (loc, scale), or with several particles of each member's
 *           brl_aggregate_predictions, into metrics[k] [M,5] = {nll, mse, sharpness, rmsce, mace};
 *      and scalars[k] [M,4] = {loss, nll_sum, kl, mse} (ELBO) or [M,2] = {loss, mse} (HNN).  Parameters and optimiser state are
 *      updated in place; no gradient is returned.  Every net, back-end and member count of the single steps runs, the same way.
 *      With step graphs on (brl_set_step_graph) and `stream` not being captured by the caller, the first step of a configuration
 *      runs eagerly, the second is captured, and every later step (this call's and a later call's with the same sizes, parameter,
 *      optimiser-state and workspace pointers and optimiser hyper-parameters beta1, beta2, eps, clip_norm, weight_decay) is one
 *      graph launch: the step reads k, the windows, the Philox key and the Adam step size from a descriptor in the workspace,
 *      which one small launch per 896 steps rewrites.  Otherwise the same launches run eagerly.  The host is never synchronised.
 *      An index outside [0, N) reads no memory: that step's rows of scalars and metrics are NaN.
 *      Workspace: brl_workspace_bytes(B, M, 5) / brl_workspace_bytes(B, M, 6); less returns BRL_ERR_WORKSPACE. */
int brl_elbo_train_steps(brl_ctx* ctx, const float* X /*[N,30,18]*/, const float* Y /*[N]*/, int64_t N, const int64_t* idx /*[K,M,B]*/,
                         int64_t K, int64_t M, int64_t B, float* loc /*[M,P]*/, float* log_scale, float* scale, float* m_loc,
                         float* v_loc, float* m_log_scale, float* v_log_scale, int64_t step0, float lr, float beta1, float beta2,
                         float eps, float clip_norm, float lrd, float weight_decay, int mode, int guide, int particles,
                         float prior_loc, float prior_scale, int64_t dataset_size, uint64_t seed, int64_t sample0, int64_t window0,
                         double* scalars /*[K,M,4]*/, double* metrics /*[K,M,5]*/, void* workspace, size_t workspace_bytes,
                         void* stream);
int brl_hnn_train_steps(brl_ctx* ctx, const float* X /*[N,30,18]*/, const float* Y /*[N]*/, int64_t N, const int64_t* idx /*[K,M,B]*/,
                        int64_t K, int64_t M, int64_t B, float* theta /*[M,P]*/, float* exp_avg, float* exp_avg_sq, int64_t step0,
                        float lr, float beta1, float beta2, float eps, float clip_norm, float lrd, float weight_decay,
                        float p_dropout, uint64_t seed, int64_t sample0, int64_t window0, double* scalars /*[K,M,2]*/,
                        double* metrics /*[K,M,5]*/, void* workspace, size_t workspace_bytes, void* stream);
/* brl_hnn_train_steps with step 2 replaced by brl_adam (torch.optim.Adam) at Adam step step0 + k + 1: no clip, no lr decay.  The
 * data, index, seed, member, metrics and graph contract and the workspace (brl_workspace_bytes(B, M, 6)) are those of
 * brl_hnn_train_steps; a step graph captured by one of the two calls is never replayed by the other. */
int brl_hnn_train_steps_adam(brl_ctx* ctx, const float* X /*[N,30,18]*/, const float* Y /*[N]*/, int64_t N,
                             const int64_t* idx /*[K,M,B]*/, int64_t K, int64_t M, int64_t B, float* theta /*[M,P]*/, float* exp_avg,
                             float* exp_avg_sq, int64_t step0, double lr, double beta1, double beta2, double eps, double weight_decay,
                             float p_dropout, uint64_t seed, int64_t sample0, int64_t window0, double* scalars /*[K,M,2]*/,
                             double* metrics /*[K,M,5]*/, void* workspace, size_t workspace_bytes, void* stream);

/* ---- K validation batches of ONE variational BNN in one call, over a device-resident split (replaces Lightning's validation loop
 *      of validation_step, bayesian.py:168-197: svi.evaluate_loss, the kl read, bnn.predict(x, S, aggregate = S > 1) and the logged
 *      metrics, with two .item() reads per batch).  X [N,30,18] (16-byte aligned), Y [N]; idx [K,B] (int64, device).  Batch k does
 *      exactly, with phi = 0x9E3779B97F4A7C15 and keys mod 2^64:
 *        1. brl_elbo_step(X[idx[k]], Y[idx[k]], mode BRL_MODE_WS, compute_grads = 0, key {seed + phi (2k + 1), sample0, window0}) on the
 *           context's gemm back-end -- validation has no fit context, so it samples weights also in LRT / Flipout experiments;
 *        2. brl_sample_weights(S, key {seed + phi (2k + 2), sample0, window0}), brl_forward(BRL_MODE_WS, engine) of the S draws and,
 *           for S > 1, brl_aggregate_predictions (S = 1: sample 0 as it is);
 *        3. brl_step_metrics of that (loc, scale) against Y[idx[k]];
 *      into scalars[k] = {loss, nll_sum, kl, mse} (brl_elbo_step) and metrics[k] = {nll, mse, sharpness, rmsce, mace}.  The two keys
 *      per batch continue the reference's per-call key sequence: validation_step draws twice per batch.  loc, scale and any optimiser
 *      state are left untouched; the host is never synchronised.  Graphs as brl_elbo_train_steps: with step graphs on, the first batch
 *      of a configuration (sizes, guide, particles, S, engine, back-end, parameter and workspace pointers) runs eagerly, the second is
 *      captured and every later batch is one graph launch (a captured graph of one kind of call is never replayed by another); with
 *      brl_tc_timing or brl_tc_trace on, the tensor-core engine's batches run eagerly, with the same results.  An index outside
 *      [0, N) reads no memory: that batch's rows are NaN.  particles 1..8, S >= 1.  Workspace: brl_workspace_bytes(B, S, 7, engine);
 *      less returns BRL_ERR_WORKSPACE. */
int brl_elbo_val_steps(brl_ctx* ctx, const float* X /*[N,30,18]*/, const float* Y /*[N]*/, int64_t N, const int64_t* idx /*[K,B]*/,
                       int64_t K, int64_t B, const float* loc /*[P]*/, const float* scale /*[P]*/, int guide, int particles, int64_t S,
                       int engine, float prior_loc, float prior_scale, int64_t dataset_size, uint64_t seed, int64_t sample0,
                       int64_t window0, double* scalars /*[K,4]*/, double* metrics /*[K,5]*/, void* workspace, size_t workspace_bytes,
                       void* stream);

/* ---- deep-ensemble mixture moments (models/deepens.py:21-24), [M,n] -> [n] ------------- */
int brl_mixture_moments(const float* mu_m, const float* sigma_m, int64_t M, int64_t n, float* mu,
                        float* sigma, void* stream);

/* ---- test-time scalar metrics (bayesian.py:217-224): device double[4] =
 *      {gaussian_nll_loss(pred,y,std^2), mse, sharpness, rms_calibration_error(100 bins)} */
int brl_test_metrics(const float* pred, const float* std, const float* y, int64_t n, double* scalars,
                     void* workspace, size_t workspace_bytes, void* stream);

/* ---- the scalars logged every training / validation / test step (bayesian.py:158-166,187-197; frequentist.py:50-58,94-110):
 *      device double[5] = {gaussian_nll_loss(pred,y,std^2), mse_loss, sharpness, rms_calibration_error, mean_absolute_calibration_error}
 *      (results/metrics.py:210-213,255-274,277-297; 100 bins, prop_type "interval") from ONE pass over the batch + a
 *      100-bin coverage histogram, instead of ~30 small torch launches per step */
int brl_step_metrics(const float* pred, const float* std, const float* y, int64_t n, double* scalars,
                     void* workspace, size_t workspace_bytes, void* stream);

/* brl_step_metrics of M rows in one pass: row m of scalars [M,5] is brl_step_metrics(pred + m*n, std + m*n, y + m*n, n).
 * Workspace: M x 1024 bytes (less returns BRL_ERR_WORKSPACE). */
int brl_step_metrics_ensemble(const float* pred /*[M,n]*/, const float* std /*[M,n]*/, const float* y /*[M,n]*/, int64_t M,
                              int64_t n, double* scalars /*[M,5]*/, void* workspace, size_t workspace_bytes, void* stream);

/* ---- fused ClippedAdam over a flat buffer (pyro.optim.ClippedAdam, conf/model/bnn.yaml:6-10) */
int brl_clipped_adam(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                     int64_t step, float lr, float beta1, float beta2, float eps, float clip_norm,
                     float lrd, float weight_decay, void* stream);

/* the same for the two flat buffers of a mean-field guide in ONE launch: ClippedAdam on `loc` and on `log_scale` (the
 * unconstrained parameter behind Pyro's positive constraint, guides/radial.py:85-94), then scale = exp(log_scale) */
int brl_clipped_adam_vi(float* loc, float* log_scale, float* scale, const float* grad_loc, const float* grad_log_scale,
                        float* m_loc, float* v_loc, float* m_log_scale, float* v_log_scale, int64_t n, int64_t step, float lr,
                        float beta1, float beta2, float eps, float clip_norm, float lrd, float weight_decay, void* stream);

/* the same with the gradients multiplied by grad_scale first (before the clamp): 1 / world_size after a SUM all-reduce of the
 * data-parallel ranks' gradients (the NVLS multimem all-reduce of dist.FlatGradAllReduce has no AVG), so no separate scaling launch */
int brl_clipped_adam_vi_scaled(float* loc, float* log_scale, float* scale, const float* grad_loc, const float* grad_log_scale,
                               float* m_loc, float* v_loc, float* m_log_scale, float* v_log_scale, int64_t n, int64_t step, float lr,
                               float beta1, float beta2, float eps, float clip_norm, float lrd, float weight_decay, float grad_scale,
                               void* stream);

/* ---- torch.optim.Adam over a flat buffer (single-tensor fp32 path, amsgrad = maximize = False: the optimizer the HNN
 *      and deep-ensemble members are configured with), one step t = `step` >= 1, per element:
 *        g += weight_decay p (L2, when weight_decay != 0);  m = lerp(m, g, 1 - beta1);  v = beta2 v + (1 - beta2) g g;
 *        p -= step_size m / (sqrt(v) / bc2_sqrt + eps),  step_size = lr / (1 - beta1^t),  bc2_sqrt = sqrt(1 - beta2^t).
 *      The hyper-parameters are doubles, as the optimizer holds them: the step scalars are computed in double and every operand
 *      is rounded to float where torch rounds it; each of torch's ops is rounded on its own (no contraction across them). */
int brl_adam(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, int64_t step, double lr, double beta1,
             double beta2, double eps, double weight_decay, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BAYESRUL_B200_H */
