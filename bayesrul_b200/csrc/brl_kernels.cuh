// Parameter blocks + launch prototypes of the fp32 SIMT engine (brl_kernels.cu).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace brl {

long long launch_count();  // kernels launched by this library since load
void count_launch(int n);

// How the A operand (activations / gradients) of an implicit GEMM is gathered:
//   row m  -> (b = m / P, oh = (m % P) / Wrow, ow = (m % P) % Wrow), image = s*B + b (or b when shared)
//   col k  -> element offset koff[k] and tap displacement (dh, dw) packed in kdhw[k]
//   value  = base[image*img_stride + oh*sH + ow*sW + koff[k]]  if (oh+dh, ow+dw) inside [0,Hin)x[0,Win) else 0
struct Gather {
  const float* base0;
  const float* base1;  // second operand of dual GEMMs (== base0 for forward)
  long long img_stride;
  int per_sample;  // 0: the tensor is shared by all MC samples (the input windows x)
  int Hin, Win, sH, sW;
  const int* koff;
  const int* kdhw;  // (dh & 0xffff) | (dw << 16)
  const int* kci;   // channel of column k (sign transform)
};

enum { TRA_NONE = 0, TRA_SQUARE = 1, TRA_SIGN = 2 };
enum { TRB_NONE = 0, TRB_SQUARE = 1, TRB_MINUS_W0 = 2 };
enum { EPI_FWD_PLAIN = 0, EPI_FWD_LRT = 1, EPI_FWD_FLIPOUT = 2, EPI_DX_PLAIN = 3, EPI_DX_LRT = 4, EPI_DX_FLIPOUT = 5 };

struct NoiseRef {       // one noise stream: injected tensor or Philox
  const float* ptr;     // injected [S, B, per_window]; nullptr -> Philox
  unsigned long long seed;
  unsigned int kind, site, sample0, window0;
  // CUDA-graph replay (brl_elbo_step): the per-step part of the key lives in device memory, {seed, sample0, window0} as
  // three 64-bit words that a one-thread kernel rewrites before every launch of the captured step; nullptr = by value
  const unsigned long long* dyn;
};
#ifdef __CUDACC__
struct NoiseKey { unsigned long long seed; unsigned int sample0, window0; };
__device__ __forceinline__ NoiseKey noise_key(const NoiseRef& nz) {
  NoiseKey k{nz.seed, nz.sample0, nz.window0};
  if (nz.dyn) {
    k.seed = __ldg(nz.dyn);
    k.sample0 += (unsigned int)__ldg(nz.dyn + 1);
    k.window0 += (unsigned int)__ldg(nz.dyn + 2);
  }
  return k;
}
#endif

struct ConvGemm {
  int B, P, Wrow;  // rows per sample = B*P; Wrow = row-space width (Wout for fwd, Win for dX)
  int N, K, S;
  Gather a;
  int trA;
  const float* sign_in;  // [S,B,sign_C] flip_in signs (TRA_SIGN, EPI_DX_FLIPOUT)
  int sign_C;
  // B operand: value0 = W0[s*ws0 + kB(k) + n*nB]; value1 = tr(W1[s*ws1 + kB(k) + n*nB])
  const float* W0;
  const float* W1;
  long long ws0, ws1;
  const int* kB;  // nullptr -> k
  int nB;
  int trB;
  // forward epilogue
  const float* bias0;  // [.. + n]
  const float* bias1;
  long long bs0, bs1;  // per-sample strides of the bias pointers
  float* out;          // activation buffer (fwd) or gradient buffer (dX, accumulated with +=)
  long long out_img_stride;
  int out_P;   // positions per channel in the out buffer
  int co_off;  // channel offset inside the out buffer (concat)
  int relu, head;
  float keep;          // dropout keep probability (1 = no dropout)
  NoiseRef eps;        // LRT eps
  NoiseRef drop;       // dropout masks
  const float* sign_out;  // [S,B,N] flip_out signs
  float* sd_out;          // LRT: sqrt(var) saved for backward, compact [img][N][P] (nullable)
  const float* xin;       // EPI_DX_LRT: the layer input (same indexing as out)
  float* part;            // split-K scratch [2][B*P][N] (nullable: no split)
  int ksplit;             // filled by launch_conv_gemm
};
constexpr long long SPLITK_SCRATCH_FLOATS = 2ll * 74 * 128 * 32;

void launch_conv_gemm(const ConvGemm& p, int epi, cudaStream_t st);
void launch_splitk_epilogue(const ConvGemm& p, int epi, cudaStream_t st);  // epilogue over p.part = [2][B * P][N] partial sums
// same operator on the tensor pipe: tcgen05 kind::tf32 dual GEMM, fp32 accumulation in TMEM (brl_tc_gemm.cu)
void launch_conv_gemm_tc(const ConvGemm& p, int epi, cudaStream_t st);
int tc_gemm_status();  // 0 ok, else code of the first mbarrier wait that timed out in a TF32 kernel (synchronises)

// weight-gradient GEMM: C[co][k] (+)= sum_m G[m][co] * tr(A[m][k]);  k == K is the bias column (A = 1)
struct ConvDw {
  int B, P, Wrow, N /*Cout*/, K;
  Gather a;
  int trA;
  const float* sign_in;
  int sign_C;
  const float* G;  // compact [img][N][P]
  float* gw;       // flat gradient buffer: gw[w_off + co*K + k]
  float* gb;       // bias gradient: gb[co] (nullable)
  float* gb2;      // second bias destination (flipout), nullable
  // optional second contraction sharing the gather (fp32 SIMT kernel only): C1[co][k] += sum_m G1[m][co] * tr1(A[m][k]),
  // i.e. the sigma^2-path (tr1 = square) or perturbation-path (tr1 = sign flip) gradient of the same layer; trA must be NONE
  const float* G1;  // nullptr -> single contraction
  int trA1;
  float* gw1;
  float* gb1;  // nullable
};
void launch_conv_dw(const ConvDw& p, cudaStream_t st);
void launch_conv_dw_tc(const ConvDw& p, cudaStream_t st);

struct PoolParams {
  const float* in;
  float* out;
  long long in_img_stride, out_img_stride;
  int C, Hin, Win, Hout;  // out is [C][Hout][Win] dense
  int sC, sH, sW;         // input strides
  long long n_img;
};
void launch_maxpool3(const PoolParams& p, cudaStream_t st);                                 // k3 s1 p1 along H
void launch_maxpool3_bwd(const PoolParams& p, const float* gout, float* gin, cudaStream_t st);  // gin += routed gout
void launch_avgpool2(const PoolParams& p, cudaStream_t st);                                 // (2,1) along H, floor
void launch_avgpool2_bwd(const PoolParams& p, const float* gout, float* gin, cudaStream_t st);

// backward through activation/dropout/head of one layer: produces compact dpre (+ dvar / dpert)
struct BwdAct {
  const float* gout;  // gradient buffer of the op output (concat layout)
  const float* outv;  // forward output (same layout)
  long long img_stride;
  int out_P, co_off, N, P;
  long long n_img;  // S*B
  int B;
  int relu, head;
  float inv_keep;
  float* dpre;  // compact [img][N][P]
  // LRT
  float* dvar;
  const float* sd;
  NoiseRef eps;
  // flipout
  float* dpert;
  const float* sign_out;
};
void launch_bwd_act(const BwdAct& p, cudaStream_t st);

// S draws [S,P]: draw s reads mu / sigma + ((s + phase) / per) mu_stride (mu_stride 0: S draws of one posterior; P with per 1:
// one draw from each of S posteriors, the members of an ensemble step; P with per > 1: `per` draws per posterior, the first
// posterior already `phase` draws in, a chunk of the member-major sample axis of brl_predict_moments_ensemble) and MC-sample
// index / injected noise row sample0 + s sample_stride
void launch_sample_normal(const float* mu, const float* sigma, long long P, long long S, NoiseRef eps, float* w,
                          float* delta, cudaStream_t st, long long mu_stride = 0, int sample_stride = 1, int per = 1,
                          int phase = 0);
void launch_sample_radial(const float* mu, const float* sigma, long long P, long long S, const long long* site_off,
                          int n_sites, int max_site, NoiseRef eps, NoiseRef r, float* norms /*[S,n_sites]*/, float* w,
                          float* delta, cudaStream_t st, long long mu_stride = 0, int sample_stride = 1, int per = 1,
                          int phase = 0);
void launch_gen_signs(float* dst, long long S, long long B, int C, NoiseRef nz, cudaStream_t st);
// all sign tensors of one particle in ONE launch (a Flipout step needs 2 per layer): job j fills dst[j][B][C[j]] with stream
// (kind[j], site[j]) of the key in `base`; with `members` > 1, member m fills dst[j][m][B][C[j]] with MC-sample index
// sample0 + m sample_stride
struct SignJobs {
  float* dst[32];
  int C[32];
  unsigned int kind[32], site[32];
  long long start[33];  // offsets of the jobs in the launch's index space (work item = four consecutive channels of a window)
  int n;
};
void launch_gen_signs_multi(const SignJobs& jobs, long long B, NoiseRef base, cudaStream_t st, int members = 1,
                            int sample_stride = 1);

void launch_nll_elbo(const float* out, const float* y, long long B, float gscale, double* acc /*[nll, mse]*/,
                     float* gout, cudaStream_t st);
void launch_nll_hnn(const float* out, const float* y, long long B, double* acc /*[loss, mse]*/, float* gout,
                    cudaStream_t st);
// analytic / sampled KL + gradient finalisation
struct Finalize {
  long long P;
  int mode, guide, first;  // first particle: write, else accumulate
  const float *mu, *sigma, *w, *delta, *g0, *g1;
  float prior_loc, prior_scale, c_kl;  // c_kl = c / particles
  float *grad_mu, *grad_sigma;
  float* grad_log_sigma;  // last particle only (nullable): d/d(log sigma) = d/d(sigma) * sigma of the summed gradient
  double* kl_acc;  // += KL (unscaled) of this particle
  // members > 1 (ensemble step): member m's mu / sigma / w / delta / g0 / g1 / grad_* sit m P floats further, its KL at
  // kl_acc + m kl_stride
  int members, kl_stride;
};
void launch_finalize(const Finalize& p, cudaStream_t st);
// scalars [members][4] from acc [members][4]
void launch_post_scalars(double* scalars, const double* acc, double c_nll, double c, int particles, long long B,
                         cudaStream_t st, int members = 1);
void launch_log_sigma_grad(const float* gs, const float* sigma, float* gls, long long P, cudaStream_t st);

void launch_moments_update(const float* out, long long S, long long B, float* state /*[4,B]*/, int first,
                           cudaStream_t st);
void launch_moments_final(const float* state, long long B, float* pred, float* std, float* ep, float* al,
                          cudaStream_t st);
// brl_predict_moments_ensemble: the Welford update of samples [j0, j0 + sc) of the member-major sample axis j = m S + s (out
// [sc,B,2]) into state [M,4,B], and the final moments of all members, out [4,M,B] = (pred, std, ep_var, al_var)
void launch_moments_update_members(const float* out, long long j0, long long sc, long long S, long long B, float* state,
                                   cudaStream_t st);
void launch_moments_final_members(const float* state, long long M, long long B, float* out, cudaStream_t st);
void launch_moments_direct(const float* out, long long S, long long B, float* pred, float* std, float* ep, float* al,
                           cudaStream_t st);
void launch_aggregate(const float* out, long long S, long long B, float* agg, cudaStream_t st);
// the aggregates of `members` members in one launch: member m's S outputs at out + m S B 2 (out [members S,B,2]) -> agg [members,B,2]
void launch_aggregate(const float* out, long long S, long long B, float* agg, cudaStream_t st, int members);
void launch_mixture(const float* mu_m, const float* sd_m, long long M, long long n, float* mu, float* sd,
                    cudaStream_t st);
// members > 1: row m of pred / std / y [members,n] -> scalars + m nscal, with the m-th 1024 bytes of the scratch at `hist`
void launch_test_metrics(const float* pred, const float* std, const float* y, long long n, double* scalars,
                         unsigned int* hist, cudaStream_t st, int nscal = 4, int members = 1);
void launch_clipped_adam(float* p, const float* g, float* m, float* v, long long n, float step_size, float b1,
                         float b2, float eps, float clip, float wd, cudaStream_t st);
void launch_clipped_adam_vi(float* loc, float* ls, float* scale, const float* g_loc, const float* g_ls, float* m_loc, float* v_loc,
                            float* m_ls, float* v_ls, long long n, float step_size, float b1, float b2, float eps, float clip, float wd,
                            cudaStream_t st, float gscale = 1.0f);  // gscale: multiplies the gradients first (1 / world after a SUM all-reduce)


// ---- K training steps per call (brl_elbo_train_steps / brl_hnn_train_steps) ----
constexpr int TRAIN_TABLE = 896;  // Adam step sizes one setup launch brings (its arguments stay below 4 KB)
// the call's descriptor in device memory: everything a replayed step reads that changes from step to step or call to call
struct TrainDesc {
  const float* X;  // [N,30,18]
  const float* Y;  // [N]
  const long long* idx;  // [K,M,B]
  double* scalars;  // [K,M,nscal]
  double* metrics;  // [K,M,5]
  long long N, k;   // k: the step being run
  int kt, bad;      // kt: step k's entry of `steps`; bad: step k's gather met an index outside [0, N)
  unsigned long long seed, sample0, window0;
  unsigned long long dyn[4];  // step k's Philox key {seed + 0x9E3779B97F4A7C15 (k + 1), sample0, window0} (NoiseRef::dyn)
  float steps[TRAIN_TABLE];   // Adam step sizes of steps k - kt ...
};
struct TrainSetup {
  TrainDesc* d;
  const float *X, *Y;
  const long long* idx;
  double *scalars, *metrics;
  long long N, k0;  // k0: first step of this table
  unsigned long long seed, sample0, window0;
  int n;
  float steps[TRAIN_TABLE];
};
void launch_train_setup(const TrainSetup& s, cudaStream_t st);
void launch_train_gather(TrainDesc* d, float* xb, float* yb, long long MB, cudaStream_t st);
// brl_elbo_val_steps{,_ensemble}: the gather of step k (idx [K,B]) into each of M member slots, xb [M,B,30,18] and yb [M,B]; it writes
// the ELBO's Philox key {seed + 0x9E3779B97F4A7C15 (2k + 1), sample0, window0} to d->dyn and the predictive draw's
// {seed + 0x9E3779B97F4A7C15 (2k + 2), sample0, window0} to key2 [4]
void launch_val_gather(TrainDesc* d, float* xb, float* yb, long long B, int M, unsigned long long* key2, cudaStream_t st);
void launch_split_pred(const float* src, long long mstride, int M, long long B, float* pred, float* std, cudaStream_t st);
void launch_train_tail(TrainDesc* d, const double* scal, int nscal, const double* met, int M, cudaStream_t st);
// ClippedAdam with the step size d->steps[d->kt] read on the device
void launch_clipped_adam(float* p, const float* g, float* m, float* v, long long n, const TrainDesc* d, float b1, float b2, float eps,
                         float clip, float wd, cudaStream_t st);
void launch_clipped_adam_vi(float* loc, float* ls, float* scale, const float* g_loc, const float* g_ls, float* m_loc, float* v_loc,
                            float* m_ls, float* v_ls, long long n, const TrainDesc* d, float b1, float b2, float eps, float clip,
                            float wd, cudaStream_t st);

// ---- torch.optim.Adam (brl_adam / brl_hnn_train_steps_adam) ----
// its float operands, each the float torch rounds its Python double to: w1 = 1 - beta1 (the lerp weight), b2 = beta2,
// w2 = 1 - beta2 (the addcmul value), eps, wd = weight_decay
struct AdamArgs {
  float w1, b2, w2, eps, wd;
};
// one step with step_size = lr / (1 - beta1^t) and bc2_sqrt = sqrt(1 - beta2^t) from the host ...
void launch_adam(float* p, const float* g, float* m, float* v, long long n, float step_size, float bc2_sqrt, const AdamArgs& a,
                 cudaStream_t st);
// ... or step k's pair d->steps[d->kt], bc2[d->kt] read on the device
void launch_adam(float* p, const float* g, float* m, float* v, long long n, const TrainDesc* d, const float* bc2, const AdamArgs& a,
                 cudaStream_t st);
// the setup launch of brl_hnn_train_steps_adam: TrainSetup (step sizes in `steps`) plus the sqrt(1 - beta2^t) column, which goes to
// `bc2` [TRAIN_TABLE] in the workspace.  Its arguments take 7.3 KB: above the 4 KB of old toolkits, within the 32 764 bytes that
// CUDA 12.1+ allows a kernel on Volta and newer.
struct TrainSetupAdam {
  TrainSetup s;
  float* bc2;
  float bc2_tab[TRAIN_TABLE];
};
static_assert(sizeof(TrainSetupAdam) <= 32764, "train_setup_adam_kernel's arguments exceed the kernel parameter limit");
void launch_train_setup(const TrainSetupAdam& s, cudaStream_t st);

}  // namespace brl
