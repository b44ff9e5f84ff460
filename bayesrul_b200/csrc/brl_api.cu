// C ABI (include/bayesrul_b200.h) + host-side tape executor of the fp32 SIMT engine.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstddef>
#include <cstdint>
#include <cstring>
#include <stdexcept>
#include <list>
#include <string>
#include <vector>

#include "../../include/bayesrul_b200.h"
#include "brl_kernels.cuh"
#include "brl_nets.h"
#include "brl_philox.cuh"
#include "brl_tc.cuh"
#include "brl_tc_train.cuh"

using namespace brl;

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define BRL_REQUIRE(cond, msg) \
  do {                         \
    if (!(cond)) return fail(BRL_ERR_INVALID, std::string("bayesrul_b200: ") + msg); \
  } while (0)
#define BRL_CUDA(expr)                                                                                   \
  do {                                                                                                   \
    cudaError_t e__ = (expr);                                                                            \
    if (e__ != cudaSuccess)                                                                              \
      return fail(BRL_ERR_CUDA, std::string("bayesrul_b200: CUDA error: ") + cudaGetErrorString(e__) + " at " #expr); \
  } while (0)

// Every entry point that takes a context runs on the context's device whatever the caller's current device is, and
// leaves the caller's current device as it found it (two Engines on two GPUs in one process; torch.cuda.set_device later on).
struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) switched = cudaSetDevice(dev) == cudaSuccess;
  }
  ~DeviceGuard() {
    if (switched) cudaSetDevice(prev);
  }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
};

// per-conv-op device tables
struct OpTables {
  int *koff = nullptr, *kdhw = nullptr, *kci = nullptr;          // forward / dW gather
  int *koff_dx = nullptr, *kdhw_dx = nullptr, *kB_dx = nullptr;  // dX gather + transposed weight offsets
};

struct brl_ctx {
  int net_id = 0, device = 0;
  int gemm_backend = BRL_GEMM_SIMT_FP32;  // per-layer GEMM back-end of brl_forward (SIMT engine) / brl_elbo_step / brl_hnn_step
  const NetSpec* net = nullptr;
  std::vector<OpTables> tabs;
  long long* site_off_dev = nullptr;
  int max_site = 0;
  int* table_pool = nullptr;
  TcState* tc = nullptr;
  // The per-layer kernels of a 256-window training batch fill a fraction of the GPU each, so independent ops run
  // concurrently: ops of one dependency level of the forward tape go to different streams, and the weight-gradient
  // kernels of the backward pass leave the critical dX chain for side streams (fork / join with events; capturable).
  // The particles of a multi-particle ELBO step are independent until their gradients are summed, so two of them run side
  // by side in two LANES (each a main stream + three side streams + its own activation / gradient buffers).
  struct Lane {
    cudaStream_t main = nullptr;  // lane 0: the caller's stream of the current call; lane 1: owned
    cudaStream_t side[3] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ev_join[3] = {nullptr, nullptr, nullptr}, ev_op[8] = {};
    cudaStream_t zero = nullptr;    // the gradient buffers are cleared here, underneath the forward pass
    cudaEvent_t ev_zero = nullptr;
  };
  std::vector<int> op_level;
  int n_levels = 0;
  bool multi_stream = true;
  Lane lanes[2];
  cudaStream_t lane1_main = nullptr;
  cudaEvent_t ev_lane_fork = nullptr, ev_lane_join = nullptr;
  // brl_predict_moments_host: the batch travels in window chunks on `copy` while the previous chunk is computed
  cudaStream_t copy = nullptr;
  cudaEvent_t ev_copy_start = nullptr, ev_chunk[8] = {};
  // CUDA-graph replay of brl_elbo_step (native Philox noise only): a step is ~60-110 small launches + event fork / joins,
  // i.e. 0.5 ms (LRT) to 1.7 ms (Flipout, 2 particles) of host enqueue time -- more than the GPU needs to run it.
  // The second call with the same key captures the step (on `cap`, since the caller's stream may be the legacy default
  // stream) over staging buffers in the caller's workspace; later calls replay it.
  struct StepKey {
    long long B, dataset_size;
    int mode, guide, particles, compute_grads, backend, has_log_sigma, members;
    float prior_loc, prior_scale;
    const void *mu, *sigma, *ws;
    size_t ws_bytes;
    // brl_elbo_train_steps / brl_hnn_train_steps / brl_hnn_train_steps_adam (train = 5 / 6 / 7; 0: a single step): the step's
    // optimizer operands ({beta1, beta2, eps, clip_norm, weight_decay}; torch's Adam: AdamArgs) and its other state buffers, baked
    // into the captured optimizer launch
    int train;
    float opt[5];
    const void* state[5];
    // brl_elbo_val_steps (train = 8; mode WS, no gradients): the predictive's MC samples and engine
    long long S;
    int engine;
    bool operator==(const StepKey& o) const {
      return B == o.B && dataset_size == o.dataset_size && mode == o.mode && guide == o.guide && particles == o.particles &&
             compute_grads == o.compute_grads && backend == o.backend && has_log_sigma == o.has_log_sigma && members == o.members &&
             prior_loc == o.prior_loc && prior_scale == o.prior_scale && mu == o.mu && sigma == o.sigma && ws == o.ws &&
             ws_bytes == o.ws_bytes && train == o.train && !memcmp(opt, o.opt, sizeof(opt)) && !memcmp(state, o.state, sizeof(state)) &&
             S == o.S && engine == o.engine;
    }
  };
  struct StepGraph { StepKey key; cudaGraphExec_t exec = nullptr; int seen = 0, launches = 0; bool bad = false; };
  std::list<StepGraph> graphs;
  bool graph_enabled = true;
  cudaStream_t cap = nullptr;
};

// bump allocator over the caller's workspace (256-byte aligned); base == nullptr only measures
struct Carve {
  char* base;
  size_t cap, used = 0;
  bool ok = true;
  Carve(void* b, size_t c) : base((char*)b), cap(c) {}
  template <typename T>
  T* take(long long n) {
    const size_t bytes = ((size_t)(n < 0 ? 0 : n) * sizeof(T) + 255) & ~(size_t)255;
    T* p = base ? reinterpret_cast<T*>(base + used) : nullptr;
    used += bytes;
    if (base && used > cap) ok = false;
    return p;
  }
};

struct ActBufs {
  std::vector<float*> act, grad, sd;  // per buffer / per buffer / per op
  std::vector<float*> dpre, dsec;  // per op: gradient w.r.t. the pre-activation / the variance or perturbation path
  float* part[4] = {nullptr, nullptr, nullptr, nullptr};  // split-K scratch, one per concurrent stream
  float *g0 = nullptr, *g1 = nullptr, *wsamp = nullptr, *delta = nullptr, *norms = nullptr;
  std::vector<float*> sgn_in, sgn_out;  // per layer
  double* acc = nullptr;
  // staging of a captured ELBO step: the graph reads / writes these, plain copies connect them to the caller's tensors
  float *st_x = nullptr, *st_y = nullptr, *st_out = nullptr, *st_gmu = nullptr, *st_gsig = nullptr, *st_glog = nullptr;
  double* st_scal = nullptr;
  unsigned long long* dyn = nullptr;
  // images of one particle lane of the level-fused tcgen05 training kernels (brl_tc_train*.cu), one set per net: `tt` for the
  // Inception conv stack, `tl` for the Linear net, `tc3` for the Conv-D3 net (the latter two carved last, only where they fit)
  TtLane tt{};
  TlLane tl{};
  Tc3Lane tc3{};
  bool fused = false;         // this net's images were carved
  int fused_members = 1;      // brl_hnn_step_ensemble / brl_elbo_step_ensemble: members whose lanes sit back to back from `tt`,
                              // fused_stride bytes apart
  long long fused_stride = 0;
};
constexpr int GRAPH_MAX_PARTICLES = 8;

static void carve_forward(const NetSpec& n, Carve& c, long long B, long long S, ActBufs& ab) {
  ab.act.resize(n.bufs.size());
  for (size_t i = 0; i < n.bufs.size(); ++i) ab.act[i] = c.take<float>((n.bufs[i].shared ? B : S * B) * n.bufs[i].elems());
}
static void carve_train(const NetSpec& n, Carve& c, long long B, ActBufs& ab) {
  ab.grad.resize(n.bufs.size());
  for (size_t i = 0; i < n.bufs.size(); ++i) ab.grad[i] = n.bufs[i].shared ? nullptr : c.take<float>(B * n.bufs[i].elems());
  ab.sd.assign(n.ops.size(), nullptr);
  ab.dpre.assign(n.ops.size(), nullptr);
  ab.dsec.assign(n.ops.size(), nullptr);
  for (size_t i = 0; i < n.ops.size(); ++i)
    if (n.ops[i].kind == OP_CONV) {
      const long long e = n.layers[n.ops[i].layer].out_elems;
      ab.sd[i] = c.take<float>(B * e);
      ab.dpre[i] = c.take<float>(B * e);  // per op, so the weight-gradient kernels can run behind the dX chain
      ab.dsec[i] = c.take<float>(B * e);
    }
  ab.g0 = c.take<float>(n.P);
  ab.g1 = c.take<float>(n.P);
  ab.wsamp = c.take<float>(n.P);
  ab.delta = c.take<float>(n.P);
  ab.norms = c.take<float>(2 * n.layers.size());
  ab.sgn_in.resize(n.layers.size());
  ab.sgn_out.resize(n.layers.size());
  for (size_t l = 0; l < n.layers.size(); ++l) {
    ab.sgn_in[l] = c.take<float>(B * n.layers[l].cin);
    ab.sgn_out[l] = c.take<float>(B * n.layers[l].cout);
  }
  ab.acc = c.take<double>(8);
  for (int i = 0; i < 4; ++i) ab.part[i] = c.take<float>(SPLITK_SCRATCH_FLOATS);
  ab.st_x = c.take<float>(B * 540);
  ab.st_y = c.take<float>(B);
  ab.st_out = c.take<float>(GRAPH_MAX_PARTICLES * B * 2);
  ab.st_gmu = c.take<float>(n.P);
  ab.st_gsig = c.take<float>(n.P);
  ab.st_glog = c.take<float>(n.P);
  ab.st_scal = c.take<double>(4);
  ab.dyn = c.take<unsigned long long>(4);
  if (n.id == BRL_NET_INCEPTION) {
    unsigned char* base = c.take<unsigned char>((long long)tt_lane_bytes(B));
    if (base) tt_carve(base, B, ab.tt);
    ab.fused = base != nullptr;
  }
}

// images of the Linear / Conv-D3 nets' fused training kernels, behind everything else of the workspace: a workspace sized for the
// per-layer kernels alone keeps its layout, and a step whose workspace has no room for them runs the per-layer kernels
static void carve_tl(const NetSpec& n, Carve& c, long long B, ActBufs& ab) {
  if (n.id != BRL_NET_LINEAR && n.id != BRL_NET_CONV) return;
  const bool lin = n.id == BRL_NET_LINEAR;
  const size_t bytes = ((size_t)(lin ? tl_lane_bytes(B) : tc3_lane_bytes(B)) + 255) & ~(size_t)255;
  if (c.base && (!c.ok || c.used + bytes > c.cap)) return;
  unsigned char* base = c.take<unsigned char>((long long)bytes);
  if (base && lin) tl_carve(base, B, ab.tl);
  if (base && !lin) tc3_carve(base, B, ab.tc3);
  ab.fused = base != nullptr;
}

// brl_hnn_step_ensemble / brl_elbo_step_ensemble (elbo) on the fused Inception kernels: the other M - 1 members' lanes right
// behind lane 0 (carve_train carves it last), the members' fc-layer sums and gradients, and graph staging for M members; the ELBO
// step adds its per-member weight draws, deltas, radial norms, native sign tensors and accumulators.  A workspace without room
// for all of it keeps the layout of the single-member step, whose body then runs once per member.
static void carve_members(const NetSpec& n, Carve& c, long long B, long long M, bool elbo, ActBufs& ab) {
  if (M < 2 || n.id != BRL_NET_INCEPTION || 2 * B * 64 > SPLITK_SCRATCH_FLOATS) return;
  Carve t = c;
  t.take<unsigned char>((M - 1) * (long long)tt_lane_bytes(B));  // tt_lane_bytes is a multiple of the carve alignment
  float* part = t.take<float>(M * 2 * B * 64);
  float* dpre = t.take<float>(M * B * 64);
  float* sx = t.take<float>(M * B * 540);
  float* sy = t.take<float>(M * B);
  float* sout = t.take<float>((elbo ? GRAPH_MAX_PARTICLES : 1) * M * B * 2);
  float* sg = t.take<float>(M * n.P);
  double* ss = t.take<double>((elbo ? 4 : 2) * M);
  ActBufs e;  // the ELBO step's buffers, [M][...]
  if (elbo) {
    e.dsec.assign(1, t.take<float>(M * B * 64));
    e.g0 = t.take<float>(M * n.P);
    e.g1 = t.take<float>(M * n.P);
    e.wsamp = t.take<float>(M * n.P);
    e.delta = t.take<float>(M * n.P);
    e.norms = t.take<float>(M * 2 * (long long)n.layers.size());
    e.sgn_in.resize(n.layers.size());
    e.sgn_out.resize(n.layers.size());
    for (size_t l = 0; l < n.layers.size(); ++l) {
      e.sgn_in[l] = t.take<float>(M * B * n.layers[l].cin);
      e.sgn_out[l] = t.take<float>(M * B * n.layers[l].cout);
    }
    e.acc = t.take<double>(4 * M);
    e.st_gsig = t.take<float>(M * n.P);
    e.st_glog = t.take<float>(M * n.P);
  }
  if (c.base && (!t.ok || !ab.fused)) return;
  c = t;
  if (!c.base) return;
  ab.fused_members = (int)M;
  ab.fused_stride = (long long)tt_lane_bytes(B);
  ab.part[0] = part;  // the fc split-K sums, [M][2][B][64]
  ab.dpre[n.ops.size() - 2] = dpre;
  ab.st_x = sx; ab.st_y = sy; ab.st_out = sout; ab.st_gmu = sg; ab.st_scal = ss;
  if (elbo) {
    ab.dsec[n.ops.size() - 2] = e.dsec[0];
    ab.g0 = e.g0; ab.g1 = e.g1; ab.wsamp = e.wsamp; ab.delta = e.delta; ab.norms = e.norms;
    ab.sgn_in = e.sgn_in; ab.sgn_out = e.sgn_out;
    ab.acc = e.acc;
    ab.st_gsig = e.st_gsig; ab.st_glog = e.st_glog;
  }
}

// brl_elbo_train_steps / brl_hnn_train_steps: the call's descriptor, the gathered batch and one step's gradients, outputs, logged
// predictions, scalars and metrics, in front of the workspace of the step itself (brl_workspace_bytes codes 3 / 4, or 1 for M = 1)
struct TrainBufs {
  TrainDesc* d;
  float *xb, *yb, *g0, *g1, *g2, *out, *agg, *pred, *std;
  double *scal, *met;
  unsigned int* hist;
};
static void carve_train_steps(const NetSpec& n, Carve& c, long long M, long long B, bool elbo, TrainBufs& t) {
  t.d = c.take<TrainDesc>(1);
  t.xb = c.take<float>(M * B * 540);
  t.yb = c.take<float>(M * B);
  t.g0 = c.take<float>(M * n.P);
  t.g1 = elbo ? c.take<float>(M * n.P) : nullptr;
  t.g2 = elbo ? c.take<float>(M * n.P) : nullptr;
  t.out = c.take<float>((elbo ? GRAPH_MAX_PARTICLES : 1) * M * B * 2);
  t.agg = elbo ? c.take<float>(M * B * 2) : nullptr;
  t.pred = c.take<float>(M * B);
  t.std = c.take<float>(M * B);
  t.scal = c.take<double>((elbo ? 4 : 2) * M);
  t.met = c.take<double>(5 * M);
  t.hist = c.take<unsigned int>(256 * M);  // the step metrics' scratch, 1024 bytes per member
}

// brl_elbo_val_steps: the call's descriptor, the predictive draw's Philox key, the gathered batch and one batch's outputs ([S,B,2] of
// the predictive, or [particles,B,2] of the ELBO step before it), aggregate, logged predictions, scalars and metrics (TrainBufs
// without gradients), in front of the region that the ELBO step and then the predictive use in turn
static void carve_val_steps(Carve& c, long long B, long long S, TrainBufs& t, unsigned long long*& key2) {
  t.d = c.take<TrainDesc>(1);
  key2 = c.take<unsigned long long>(4);
  t.xb = c.take<float>(B * 540);
  t.yb = c.take<float>(B);
  t.g0 = t.g1 = t.g2 = nullptr;
  t.out = c.take<float>(std::max<long long>(GRAPH_MAX_PARTICLES, S) * B * 2);
  t.agg = c.take<float>(B * 2);
  t.pred = c.take<float>(B);
  t.std = c.take<float>(B);
  t.scal = c.take<double>(4);
  t.met = c.take<double>(5);
  t.hist = c.take<unsigned int>(256);  // the step metrics' scratch
}
// the predictive's part of that region: S weight draws [S,P], their radial norms [S,n_sites], then brl_forward's workspace
struct ValPredict {
  float *wsamp, *norms;
  size_t norms_bytes;
  char* fws;
  size_t fws_bytes;
};
static size_t carve_val_predict(const brl_ctx* ctx, Carve& c, long long B, long long S, int engine, ValPredict& v) {
  const NetSpec& n = *ctx->net;
  v.wsamp = c.take<float>(S * n.P);
  const size_t at = c.used;
  v.norms = c.take<float>(S * 2 * (long long)n.layers.size());
  v.norms_bytes = c.used - at;
  size_t fwd = tc_workspace_bytes(ctx->tc, B, S);
  if (engine != BRL_ENGINE_TC_FP16) {
    Carve f(nullptr, 0);
    ActBufs ab;
    carve_forward(n, f, B, S, ab);
    fwd = f.used;
  }
  v.fws = c.take<char>((long long)fwd);
  v.fws_bytes = fwd;
  return c.used;
}

// device {seed, sample0, window0} of the step being captured (nullptr outside a capture): every Philox stream built by
// nref() then reads the per-step part of its key from there
static thread_local const unsigned long long* g_dyn = nullptr;
// Staging of a replayed step in ONE launch per side: a few (dst, src, floats) copies (+ the Philox key on the way in) instead of a
// chain of tiny memcpy nodes on the critical path.  All pointers are 4-byte aligned device pointers.
struct CopyJobs {
  float* dst[6];
  const float* src[6];
  long long n[6], start[7];  // floats per job; offsets in the launch's index space
  int njobs;
  unsigned long long* dyn;  // nullable: {seed, sample0, window0} written by thread 0
  unsigned long long seed, sample0, window0;
};
__global__ void copy_jobs_kernel(const CopyJobs j) {
  if (j.dyn && blockIdx.x == 0 && threadIdx.x == 0) { j.dyn[0] = j.seed; j.dyn[1] = j.sample0; j.dyn[2] = j.window0; }
  const long long total = j.start[j.njobs];
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int k = 0;
    while (k + 1 < j.njobs && i >= j.start[k + 1]) ++k;
    j.dst[k][i - j.start[k]] = j.src[k][i - j.start[k]];
  }
}
static void launch_copy_jobs(CopyJobs& j, cudaStream_t st) {
  j.start[0] = 0;
  for (int k = 0; k < j.njobs; ++k) j.start[k + 1] = j.start[k] + j.n[k];
  const long long total = std::max<long long>(j.start[j.njobs], 1);
  count_launch(1);
  copy_jobs_kernel<<<(unsigned)std::min<long long>((total + 255) / 256, 148 * 8), 256, 0, st>>>(j);
}

static NoiseRef nref(const brl_noise* nz, const float* ptr, unsigned kind, unsigned site) {
  NoiseRef r;
  r.ptr = ptr;
  r.dyn = ptr ? nullptr : g_dyn;
  r.seed = nz ? nz->seed : 0ull;
  r.kind = kind;
  r.site = site;
  r.sample0 = nz ? (unsigned)nz->sample0 : 0u;
  r.window0 = nz ? (unsigned)nz->window0 : 0u;
  return r;
}

// shift every injected pointer to MC sample `s` of a call over B windows
static brl_noise noise_at_sample(const NetSpec& n, const brl_noise* nz, long long s, long long B) {
  brl_noise o;
  memset(&o, 0, sizeof(o));
  if (!nz) return o;
  o = *nz;
  o.sample0 = nz->sample0 + s;
  if (o.weight_eps) o.weight_eps += s * n.P;
  if (o.radial_r) o.radial_r += s * (long long)(2 * n.layers.size());
  for (size_t l = 0; l < n.layers.size(); ++l) {
    const LayerSpec& L = n.layers[l];
    if (o.lrt_eps[l]) o.lrt_eps[l] += s * B * L.out_elems;
    if (o.drop_mask[l]) o.drop_mask[l] += s * B * L.out_elems;
    if (o.flip_in[l]) o.flip_in[l] += s * B * L.cin;
    if (o.flip_out[l]) o.flip_out[l] += s * B * L.cout;
  }
  return o;
}

struct FwdArgs {
  const float* x;
  long long B, S;
  int mode;
  const float *theta, *sigma, *wsamp;
  float p_dropout;
  const brl_noise* noise;
  const float* const* sgn_in;   // per layer (flipout), resolved pointers
  const float* const* sgn_out;
  float* out;  // [S,B,2] or nullptr (leave in the net's output buffer)
  bool save_sd;
};

static Gather fwd_gather(const brl_ctx* ctx, const OpSpec& op, size_t oi, const ActBufs& ab, const float* x) {
  const NetSpec& n = *ctx->net;
  Gather g{};
  if (op.in.buf < 0) {
    g.base0 = x; g.img_stride = 540; g.per_sample = 0;
    g.sH = n.xsH; g.sW = n.xsW;
  } else {
    g.base0 = ab.act[op.in.buf]; g.img_stride = n.bufs[op.in.buf].elems(); g.per_sample = n.bufs[op.in.buf].shared ? 0 : 1;
    g.sH = op.in.W; g.sW = 1;
  }
  g.base1 = g.base0;
  g.Hin = op.in.H; g.Win = op.in.W;
  g.koff = ctx->tabs[oi].koff; g.kdhw = ctx->tabs[oi].kdhw; g.kci = ctx->tabs[oi].kci;
  return g;
}

static PoolParams pool_params(const NetSpec& n, const OpSpec& op, const ActBufs& ab, const float* x, long long B, long long S) {
  PoolParams p{};
  if (op.in.buf < 0) {
    p.in = x; p.in_img_stride = 540; p.sC = n.xsC; p.sH = n.xsH; p.sW = n.xsW; p.n_img = B;
  } else {
    p.in = ab.act[op.in.buf]; p.in_img_stride = n.bufs[op.in.buf].elems();
    p.sC = op.in.H * op.in.W; p.sH = op.in.W; p.sW = 1;
    p.n_img = n.bufs[op.in.buf].shared ? B : S * B;
  }
  p.out = ab.act[op.out_buf]; p.out_img_stride = n.bufs[op.out_buf].elems();
  p.C = op.in.C; p.Hin = op.in.H; p.Win = op.in.W; p.Hout = op.Hout;
  return p;
}

// operator descriptor of a conv / linear op's forward pass (operands, noise, epilogue) and its epilogue kind
static ConvGemm fwd_gemm(const brl_ctx* ctx, const ActBufs& ab, const FwdArgs& a, size_t oi, int slot, int* epi_out) {
  const NetSpec& n = *ctx->net;
  const OpSpec& op = n.ops[oi];
  const LayerSpec& L = n.layers[op.layer];
  ConvGemm p{};
  p.B = (int)a.B; p.P = op.Hout * op.Wout; p.Wrow = op.Wout; p.N = L.cout; p.K = L.cin * L.kh * L.kw; p.S = (int)a.S;
  p.a = fwd_gather(ctx, op, oi, ab, a.x);
  p.kB = nullptr; p.nB = p.K;
  int epi = EPI_FWD_PLAIN;
  switch (a.mode) {
    case BRL_MODE_DET:
      p.W0 = a.theta + L.w_off; p.bias0 = a.theta + L.b_off; break;
    case BRL_MODE_WS:
      p.W0 = a.wsamp + L.w_off; p.ws0 = n.P; p.bias0 = a.wsamp + L.b_off; p.bs0 = n.P; break;
    case BRL_MODE_LRT:
      epi = EPI_FWD_LRT;
      p.W0 = a.theta + L.w_off; p.W1 = a.sigma + L.w_off; p.trA = TRA_SQUARE; p.trB = TRB_SQUARE;
      p.bias0 = a.theta + L.b_off; p.bias1 = a.sigma + L.b_off;
      p.eps = nref(a.noise, a.noise ? a.noise->lrt_eps[op.layer] : nullptr, KIND_LRT_EPS, op.layer);
      p.sd_out = a.save_sd ? ab.sd[oi] : nullptr;
      break;
    case BRL_MODE_FLIPOUT:
      epi = EPI_FWD_FLIPOUT;
      p.W0 = a.theta + L.w_off; p.W1 = a.wsamp + L.w_off; p.ws1 = n.P; p.trA = TRA_SIGN; p.trB = TRB_MINUS_W0;
      p.sign_in = a.sgn_in[op.layer]; p.sign_C = L.cin; p.sign_out = a.sgn_out[op.layer];
      p.bias1 = a.wsamp + L.b_off; p.bs1 = n.P;
      break;
  }
  const bool is_last = op.out_buf == n.out_buf;
  p.out = (is_last && a.out) ? a.out : ab.act[op.out_buf];
  p.out_img_stride = n.bufs[op.out_buf].elems();
  p.out_P = n.bufs[op.out_buf].H * n.bufs[op.out_buf].W;
  p.co_off = op.co_off; p.relu = op.relu; p.head = op.head;
  p.keep = (a.p_dropout > 0.f && L.drop_factor > 0.f) ? 1.0f - a.p_dropout * L.drop_factor : 1.0f;
  p.drop = nref(a.noise, a.noise ? a.noise->drop_mask[op.layer] : nullptr, KIND_DROPOUT, op.layer);
  p.part = ab.part[slot];
  *epi_out = epi;
  return p;
}

static void forward_op(const brl_ctx* ctx, const ActBufs& ab, const FwdArgs& a, size_t oi, cudaStream_t st, int slot) {
  const NetSpec& n = *ctx->net;
  const OpSpec& op = n.ops[oi];
  if (op.kind == OP_MAXPOOL3) { launch_maxpool3(pool_params(n, op, ab, a.x, a.B, a.S), st); return; }
  if (op.kind == OP_AVGPOOL2) { launch_avgpool2(pool_params(n, op, ab, a.x, a.B, a.S), st); return; }
  int epi;
  const ConvGemm p = fwd_gemm(ctx, ab, a, oi, slot, &epi);
  static const int ablate = getenv("BRL_ABLATE") ? atoi(getenv("BRL_ABLATE")) : 0;
  if (ablate & 8) return;
  if ((ctx->gemm_backend & 1) && ctx->gemm_backend <= BRL_GEMM_TC_TF32) launch_conv_gemm_tc(p, epi, st);
  else launch_conv_gemm(p, epi, st);
}

static void run_forward(const brl_ctx* ctx, const ActBufs& ab, const FwdArgs& a, cudaStream_t st, int lane_id = 0) {
  const NetSpec& n = *ctx->net;
  const brl_ctx::Lane& ln = ctx->lanes[lane_id];
  // every level of the tape: ops whose inputs are complete; the first op stays on `st`, the others fork to side streams
  for (int lvl = 0; lvl < ctx->n_levels; ++lvl) {
    int cnt = 0;
    for (size_t oi = 0; oi < n.ops.size(); ++oi) cnt += ctx->op_level[oi] == lvl;
    const bool fork = ctx->multi_stream && cnt > 1;
    if (fork) cudaEventRecord(ln.ev_fork, st);  // everything the level reads is complete on `st` at this point
    int j = 0, used = 0;
    for (size_t oi = 0; oi < n.ops.size(); ++oi) {
      if (ctx->op_level[oi] != lvl) continue;
      if (j == 0 || !fork) {
        forward_op(ctx, ab, a, oi, st, 0);
      } else {
        const int si = (j - 1) % 3;
        if (!(used & (1 << si))) { cudaStreamWaitEvent(ln.side[si], ln.ev_fork, 0); used |= 1 << si; }
        forward_op(ctx, ab, a, oi, ln.side[si], 1 + si);
      }
      ++j;
    }
    for (int si = 0; si < 3; ++si)
      if (used & (1 << si)) {
        cudaEventRecord(ln.ev_join[si], ln.side[si]);
        cudaStreamWaitEvent(st, ln.ev_join[si], 0);
      }
  }
}

struct BwdArgs {
  const float* x;
  long long B;
  int mode;  // DET/WS: plain weights `w`; LRT/FLIPOUT: mu (+ sigma / wsamp)
  const float *w, *sigma, *wsamp;
  float p_dropout;
  const brl_noise* noise;
  const float* const* sgn_in;
  const float* const* sgn_out;
  const float* out;  // [B,2] forward output (the head's buffer)
  float *g0, *g1;    // flat gradient accumulators
};

// backward through the activation / dropout / head of conv op `oi`: gradient of the op output -> compact dpre (+ dvar / dpert)
static void backward_act(const brl_ctx* ctx, const ActBufs& ab, const BwdArgs& a, int oi, cudaStream_t cs) {
  const NetSpec& n = *ctx->net;
  const OpSpec& op = n.ops[oi];
  const LayerSpec& L = n.layers[op.layer];
  const int Pout = op.Hout * op.Wout;
  const bool is_last = op.out_buf == n.out_buf;
  const float keep = (a.p_dropout > 0.f && L.drop_factor > 0.f) ? 1.0f - a.p_dropout * L.drop_factor : 1.0f;
  BwdAct ba{};
  ba.gout = ab.grad[op.out_buf];
  ba.outv = (is_last && a.out) ? a.out : ab.act[op.out_buf];
  ba.img_stride = n.bufs[op.out_buf].elems();
  ba.out_P = n.bufs[op.out_buf].H * n.bufs[op.out_buf].W;
  ba.co_off = op.co_off; ba.N = L.cout; ba.P = Pout; ba.n_img = a.B; ba.B = (int)a.B;
  ba.relu = op.relu; ba.head = op.head; ba.inv_keep = 1.0f / keep;
  ba.dpre = ab.dpre[oi];
  if (a.mode == BRL_MODE_LRT) {
    ba.dvar = ab.dsec[oi]; ba.sd = ab.sd[oi];
    ba.eps = nref(a.noise, a.noise ? a.noise->lrt_eps[op.layer] : nullptr, KIND_LRT_EPS, op.layer);
  } else if (a.mode == BRL_MODE_FLIPOUT) {
    ba.dpert = ab.dsec[oi]; ba.sign_out = a.sgn_out[op.layer];
  }
  launch_bwd_act(ba, cs);
}

// expects grad[out_buf] to hold dLoss/d(out) and every other grad buffer zeroed
// backward of one op on stream `cs` (slot: 0 = the caller's stream, 1.. = side stream): activation backward, input
// gradient (the critical chain; `ev_dx`, if given, is recorded right behind it) and the weight gradients, which only
// need this op's dpre / dsec and write their own slice of the flat gradient buffers: they run on `ws`
static void backward_op(const brl_ctx* ctx, const ActBufs& ab, const BwdArgs& a, int oi, cudaStream_t cs, int slot,
                        cudaStream_t ws, cudaEvent_t ev_act, cudaEvent_t ev_dx) {
  const NetSpec& n = *ctx->net;
  const OpSpec& op = n.ops[oi];
  if (op.kind != OP_CONV) {
    if (op.in.buf >= 0) {  // (a pooled raw input needs no gradient)
      PoolParams pp = pool_params(n, op, ab, a.x, a.B, 1);
      if (op.kind == OP_MAXPOOL3) launch_maxpool3_bwd(pp, ab.grad[op.out_buf], ab.grad[op.in.buf], cs);
      else launch_avgpool2_bwd(pp, ab.grad[op.out_buf], ab.grad[op.in.buf], cs);
    }
    if (ev_dx) cudaEventRecord(ev_dx, cs);
    return;
  }
  const LayerSpec& L = n.layers[op.layer];
  const int Pout = op.Hout * op.Wout;
  static const int ablate = getenv("BRL_ABLATE") ? atoi(getenv("BRL_ABLATE")) : 0;  // timing experiments only (wrong results)
  if (!(ablate & 4)) backward_act(ctx, ab, a, oi, cs);
  if (ws != cs) {  // the weight-gradient stream picks up behind the activation backward
    cudaEventRecord(ev_act, cs);
    cudaStreamWaitEvent(ws, ev_act, 0);
  }

  // input gradient (accumulated with atomics: the ops of a level may share their input buffer)
  if (op.in.buf >= 0 && !n.bufs[op.in.buf].shared) {
    ConvGemm p{};
    p.B = (int)a.B; p.P = op.in.H * op.in.W; p.Wrow = op.in.W; p.N = L.cin; p.K = L.cout * L.kh * L.kw; p.S = 1;
    p.a.base0 = ab.dpre[oi]; p.a.base1 = ab.dsec[oi]; p.a.img_stride = (long long)L.cout * Pout; p.a.per_sample = 1;
    p.a.Hin = op.Hout; p.a.Win = op.Wout; p.a.sH = op.Wout; p.a.sW = 1;
    p.a.koff = ctx->tabs[oi].koff_dx; p.a.kdhw = ctx->tabs[oi].kdhw_dx; p.a.kci = nullptr;
    p.kB = ctx->tabs[oi].kB_dx; p.nB = L.kh * L.kw;
    p.W0 = a.w + L.w_off;
    p.out = ab.grad[op.in.buf];
    p.out_img_stride = n.bufs[op.in.buf].elems();
    p.out_P = op.in.H * op.in.W; p.co_off = 0;
    int epi = EPI_DX_PLAIN;
    if (a.mode == BRL_MODE_LRT) {
      epi = EPI_DX_LRT; p.W1 = a.sigma + L.w_off; p.trB = TRB_SQUARE; p.xin = ab.act[op.in.buf];
    } else if (a.mode == BRL_MODE_FLIPOUT) {
      epi = EPI_DX_FLIPOUT; p.W1 = a.wsamp + L.w_off; p.trB = TRB_MINUS_W0; p.sign_in = a.sgn_in[op.layer]; p.sign_C = L.cin;
    }
    p.part = ab.part[slot];
    if (ablate & 2) {}
    else if (ctx->gemm_backend & 2) launch_conv_gemm_tc(p, epi, cs);
    else launch_conv_gemm(p, epi, cs);
  }
  if (ev_dx) cudaEventRecord(ev_dx, cs);
  if (ablate & 1) return;

  // weight gradients
  ConvDw dw{};
  dw.B = (int)a.B; dw.P = Pout; dw.Wrow = op.Wout; dw.N = L.cout; dw.K = L.cin * L.kh * L.kw;
  dw.a = fwd_gather(ctx, op, oi, ab, a.x);
  dw.G = ab.dpre[oi]; dw.gw = a.g0 + L.w_off; dw.gb = a.g0 + L.b_off;
  dw.gb2 = a.mode == BRL_MODE_FLIPOUT ? a.g1 + L.b_off : nullptr;
  if (!(ctx->gemm_backend & 4) && (a.mode == BRL_MODE_LRT || a.mode == BRL_MODE_FLIPOUT)) {
    // fp32 SIMT back-end: the mean-path and the variance- / perturbation-path weight gradients share one gather
    dw.G1 = ab.dsec[oi]; dw.gw1 = a.g1 + L.w_off;
    if (a.mode == BRL_MODE_LRT) { dw.trA1 = TRA_SQUARE; dw.gb1 = a.g1 + L.b_off; }
    else { dw.trA1 = TRA_SIGN; dw.sign_in = a.sgn_in[op.layer]; dw.sign_C = L.cin; dw.gb1 = nullptr; }
    launch_conv_dw(dw, ws);
    return;
  }
  ((ctx->gemm_backend & 4) ? launch_conv_dw_tc(dw, ws) : launch_conv_dw(dw, ws));
  if (a.mode == BRL_MODE_LRT) {
    dw.G = ab.dsec[oi]; dw.trA = TRA_SQUARE; dw.gw = a.g1 + L.w_off; dw.gb = a.g1 + L.b_off; dw.gb2 = nullptr;
    ((ctx->gemm_backend & 4) ? launch_conv_dw_tc(dw, ws) : launch_conv_dw(dw, ws));
  } else if (a.mode == BRL_MODE_FLIPOUT) {
    dw.G = ab.dsec[oi]; dw.trA = TRA_SIGN; dw.sign_in = a.sgn_in[op.layer]; dw.sign_C = L.cin;
    dw.gw = a.g1 + L.w_off; dw.gb = nullptr; dw.gb2 = nullptr;
    ((ctx->gemm_backend & 4) ? launch_conv_dw_tc(dw, ws) : launch_conv_dw(dw, ws));
  }
}

// expects grad[out_buf] to hold dLoss/d(out) and every other grad buffer zeroed.  Tape levels run in reverse; the ops
// of a level run concurrently (first op on `st`, the others on side streams), the next level waits for their dX only.
static void run_backward(const brl_ctx* ctx, const ActBufs& ab, const BwdArgs& a, cudaStream_t st, int lane_id = 0) {
  const NetSpec& n = *ctx->net;
  const brl_ctx::Lane& ln = ctx->lanes[lane_id];
  if (!ctx->multi_stream) {
    for (int oi = (int)n.ops.size() - 1; oi >= 0; --oi) backward_op(ctx, ab, a, oi, st, 0, st, nullptr, nullptr);
    return;
  }
  int n_dw = 0, used_any = 0;
  for (int lvl = ctx->n_levels - 1; lvl >= 0; --lvl) {
    int cnt = 0;
    for (size_t oi = 0; oi < n.ops.size(); ++oi) cnt += ctx->op_level[oi] == lvl;
    const bool fork = cnt > 1;
    if (fork) cudaEventRecord(ln.ev_fork, st);
    int j = 0, used = 0;
    for (int oi = (int)n.ops.size() - 1; oi >= 0; --oi) {
      if (ctx->op_level[oi] != lvl) continue;
      if (j == 0) {  // on the caller's stream; its weight gradients go to a rotating side stream
        const int wi = n_dw++ % 3;
        used_any |= 1 << wi;
        backward_op(ctx, ab, a, oi, st, 0, ln.side[wi], ln.ev_op[n_dw % 8], nullptr);
      } else {
        const int si = (j - 1) % 3;
        if (!(used & (1 << si))) { cudaStreamWaitEvent(ln.side[si], ln.ev_fork, 0); used |= 1 << si; }
        backward_op(ctx, ab, a, oi, ln.side[si], 1 + si, ln.side[si], nullptr, ln.ev_join[si]);
      }
      ++j;
    }
    used_any |= used;
    for (int si = 0; si < 3; ++si)
      if (used & (1 << si)) cudaStreamWaitEvent(st, ln.ev_join[si], 0);  // the side chains' dX (recorded behind each)
  }
  for (int si = 0; si < 3; ++si)  // final join: the weight gradients too; the caller's stream owns the buffers again
    if (used_any & (1 << si)) {
      cudaEventRecord(ln.ev_join[si], ln.side[si]);
      cudaStreamWaitEvent(st, ln.ev_join[si], 0);
    }
}

static int zero_grads(const NetSpec& n, const ActBufs& ab, long long B, cudaStream_t st) {
  for (size_t i = 0; i < n.bufs.size(); ++i)
    if (ab.grad[i]) BRL_CUDA(cudaMemsetAsync(ab.grad[i], 0, sizeof(float) * B * n.bufs[i].elems(), st));
  return BRL_OK;
}

// the caller is capturing `st` itself (e.g. torch.cuda.graph): stay on the eager, capturable path
static bool stream_capturing(cudaStream_t st) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) { cudaGetLastError(); return true; }
  return cs != cudaStreamCaptureStatusNone;
}

// the context's captured step for `key` (most recently used first, at most 16), a new empty one on first sight
static brl_ctx::StepGraph* graph_slot(brl_ctx* ctx, const brl_ctx::StepKey& key) {
  for (auto it = ctx->graphs.begin(); it != ctx->graphs.end(); ++it)
    if (it->key == key) { ctx->graphs.splice(ctx->graphs.begin(), ctx->graphs, it); return &ctx->graphs.front(); }
  if (ctx->graphs.size() >= 16) {
    if (ctx->graphs.back().exec) cudaGraphExecDestroy(ctx->graphs.back().exec);
    ctx->graphs.pop_back();
  }
  ctx->graphs.emplace_front();
  ctx->graphs.front().key = key;
  return &ctx->graphs.front();
}

// captures issue(stream) into sg (on `cap`, since the caller's stream may be the legacy default stream), every Philox stream
// reading the per-step part of its key from `dyn`; a failed capture marks sg bad, and the caller stays eager
template <class Issue>
static void capture_step(brl_ctx* ctx, brl_ctx::StepGraph* sg, const unsigned long long* dyn, Issue issue) {
  cudaGraph_t graph = nullptr;
  if (cudaStreamBeginCapture(ctx->cap, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
    g_dyn = dyn;
    const long long l0 = launch_count();
    const int rc = issue(ctx->cap);
    g_dyn = nullptr;
    sg->launches = (int)(launch_count() - l0);
    count_launch(-sg->launches);  // captured, not executed
    const cudaError_t e = cudaStreamEndCapture(ctx->cap, &graph);
    if (rc != BRL_OK || e != cudaSuccess || !graph || cudaGraphInstantiate(&sg->exec, graph, 0) != cudaSuccess) {
      sg->exec = nullptr;
      sg->bad = true;
    }
    if (graph) cudaGraphDestroy(graph);
  } else {
    sg->bad = true;
  }
  cudaGetLastError();  // a failed capture must not poison the eager path
}

// Graph replay of a training step whose configuration is `key`, where `graphable` (native Philox noise): eager on first sight of
// the key, captured on the second, replayed after.  body(x, y, noise, staged, stream) issues the step's launches; `staged` selects
// the outputs among ab's staging buffers instead of the caller's.  The capture runs it over the staging inputs with the Philox key
// read from ab.dyn; a replay copies x, y (MB windows) and the key in, launches the graph and copies `out` back.
template <class Body>
static int run_step(brl_ctx* ctx, const brl_ctx::StepKey& key, bool graphable, const ActBufs& ab, const float* x, const float* y,
                    long long MB, const brl_noise* noise, CopyJobs out, Body body, cudaStream_t st) {
  brl_ctx::StepGraph* sg = nullptr;
  if (ctx->graph_enabled && graphable && !stream_capturing(st)) {
    sg = graph_slot(ctx, key);
    ++sg->seen;
    if (sg->seen >= 2 && !sg->exec && !sg->bad)
      capture_step(ctx, sg, ab.dyn, [&](cudaStream_t cs) {
        brl_noise zero;
        memset(&zero, 0, sizeof(zero));
        return body(ab.st_x, ab.st_y, &zero, true, cs);
      });
  }
  if (!sg || !sg->exec) return body(x, y, noise, false, st);
  count_launch(sg->launches);
  CopyJobs in{};  // x, y and the Philox key of this step -> staging
  in.dst[0] = ab.st_x; in.src[0] = x; in.n[0] = MB * 540;
  in.dst[1] = ab.st_y; in.src[1] = y; in.n[1] = MB;
  in.njobs = 2;
  in.dyn = ab.dyn;
  in.seed = noise ? noise->seed : 0ull;
  in.sample0 = noise ? (unsigned long long)noise->sample0 : 0ull;
  in.window0 = noise ? (unsigned long long)noise->window0 : 0ull;
  launch_copy_jobs(in, st);
  BRL_CUDA(cudaGraphLaunch(sg->exec, st));
  launch_copy_jobs(out, st);
  BRL_CUDA(cudaGetLastError());
  return BRL_OK;
}

// the step size of ClippedAdam step `step` (>= 1): lr lrd^step sqrt(1 - beta2^step) / (1 - beta1^step), in double, rounded once
static float adam_step_size(float lr, float lrd, float beta1, float beta2, long long step) {
  const double lr_t = (double)lr * std::pow((double)lrd, (double)step);
  const double bc1 = 1.0 - std::pow((double)beta1, (double)step), bc2 = 1.0 - std::pow((double)beta2, (double)step);
  return (float)(lr_t * std::sqrt(bc2) / bc1);
}

// torch.optim.Adam's per-step scalars of step `step` (>= 1), as Python computes them in double from the hyper-parameters the
// optimizer holds: step_size = lr / (1 - beta1^step) and bc2_sqrt = sqrt(1 - beta2^step), each rounded once to the float its
// kernel receives
static void torch_adam_step(double lr, double beta1, double beta2, long long step, float* step_size, float* bc2_sqrt) {
  *step_size = (float)(lr / (1.0 - std::pow(beta1, (double)step)));
  *bc2_sqrt = (float)std::sqrt(1.0 - std::pow(beta2, (double)step));
}
// and its step-independent float operands (1 - beta1 and 1 - beta2 are taken in double first, as in Python)
static AdamArgs torch_adam_args(double beta1, double beta2, double eps, double weight_decay) {
  return AdamArgs{(float)(1.0 - beta1), (float)beta2, (float)(1.0 - beta2), (float)eps, (float)weight_decay};
}

// ------------------------------------------------------------------------------------------------
extern "C" {

int brl_version(void) { return 100; }
int64_t brl_launch_count(void) { return (int64_t)launch_count(); }
const char* brl_last_error(void) { return g_err.c_str(); }

int brl_net_num_params(int net) { try { return (int)get_net(net).P; } catch (...) { return BRL_ERR_INVALID; } }
int brl_net_num_layers(int net) { try { return (int)get_net(net).layers.size(); } catch (...) { return BRL_ERR_INVALID; } }
int brl_net_num_sites(int net) { try { return 2 * (int)get_net(net).layers.size(); } catch (...) { return BRL_ERR_INVALID; } }
int64_t brl_net_flops_fwd(int net) { try { return get_net(net).flops_fwd; } catch (...) { return BRL_ERR_INVALID; } }

int brl_net_site(int net, int site, int64_t* offset, int* ndim, int64_t shape[4]) {
  try {
    const NetSpec& n = get_net(net);
    BRL_REQUIRE(site >= 0 && site < 2 * (int)n.layers.size(), "site out of range");
    const LayerSpec& L = n.layers[site / 2];
    for (int i = 0; i < 4; ++i) shape[i] = 1;
    if (site % 2 == 0) {
      *offset = L.w_off; *ndim = L.wndim;
      for (int i = 0; i < L.wndim; ++i) shape[i] = L.wshape[i];
    } else {
      *offset = L.b_off; *ndim = 1; shape[0] = L.cout;
    }
    return BRL_OK;
  } catch (...) { return fail(BRL_ERR_INVALID, "unknown net"); }
}

int brl_net_layer(int net, int layer, int* cout, int* cin, int* out_elems, float* dropout_factor) {
  try {
    const NetSpec& n = get_net(net);
    BRL_REQUIRE(layer >= 0 && layer < (int)n.layers.size(), "layer out of range");
    const LayerSpec& L = n.layers[layer];
    *cout = L.cout; *cin = L.cin; *out_elems = L.out_elems; *dropout_factor = L.drop_factor;
    return BRL_OK;
  } catch (...) { return fail(BRL_ERR_INVALID, "unknown net"); }
}

int brl_create(brl_ctx** out, int net, int device) {
  BRL_REQUIRE(out != nullptr, "ctx pointer is NULL");
  const NetSpec* ns;
  try { ns = &get_net(net); } catch (...) { return fail(BRL_ERR_INVALID, "unknown net"); }
  int ndev = 0;
  BRL_CUDA(cudaGetDeviceCount(&ndev));
  BRL_REQUIRE(device >= 0 && device < ndev, "device index out of range");
  cudaDeviceProp prop;
  BRL_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(BRL_ERR_UNSUPPORTED, "bayesrul_b200: built for sm_100a (B200) only; device is sm_" +
                                         std::to_string(prop.major) + std::to_string(prop.minor) + " -- no fallback by design");
  DeviceGuard dg(device);  // restored on return: creating a context does not change the caller's current device
  brl_ctx* c = new brl_ctx();
  c->net_id = net; c->device = device; c->net = ns;
  // build gather tables
  std::vector<int> pool;
  struct Loc { size_t koff, kdhw, kci, koff_dx, kdhw_dx, kB_dx; };
  std::vector<Loc> locs(ns->ops.size());
  for (size_t oi = 0; oi < ns->ops.size(); ++oi) {
    const OpSpec& op = ns->ops[oi];
    if (op.kind != OP_CONV) continue;
    const LayerSpec& L = ns->layers[op.layer];
    int sC, sH, sW;
    if (op.in.buf < 0) { sC = ns->xsC; sH = ns->xsH; sW = ns->xsW; }
    else { sC = op.in.H * op.in.W; sH = op.in.W; sW = 1; }
    const int KK = L.kh * L.kw, K = L.cin * KK, Kdx = L.cout * KK, Pout = op.Hout * op.Wout;
    Loc lc;
    lc.koff = pool.size();
    for (int k = 0; k < K; ++k) { int ci = k / KK, r = k % KK, kh = r / L.kw, kw = r % L.kw; pool.push_back(ci * sC + (kh - L.ph) * sH + (kw - L.pw) * sW); }
    lc.kdhw = pool.size();
    for (int k = 0; k < K; ++k) { int r = k % KK, kh = r / L.kw, kw = r % L.kw; pool.push_back(((kh - L.ph) & 0xffff) | ((kw - L.pw) << 16)); }
    lc.kci = pool.size();
    for (int k = 0; k < K; ++k) pool.push_back(k / KK);
    lc.koff_dx = pool.size();
    for (int k = 0; k < Kdx; ++k) { int co = k / KK, r = k % KK, kh = r / L.kw, kw = r % L.kw; pool.push_back(co * Pout + (L.ph - kh) * op.Wout + (L.pw - kw)); }
    lc.kdhw_dx = pool.size();
    for (int k = 0; k < Kdx; ++k) { int r = k % KK, kh = r / L.kw, kw = r % L.kw; pool.push_back(((L.ph - kh) & 0xffff) | ((L.pw - kw) << 16)); }
    lc.kB_dx = pool.size();
    for (int k = 0; k < Kdx; ++k) { int co = k / KK, r = k % KK; pool.push_back(co * L.cin * KK + r); }
    locs[oi] = lc;
  }
  BRL_CUDA(cudaMalloc(&c->table_pool, pool.size() * sizeof(int)));
  BRL_CUDA(cudaMemcpy(c->table_pool, pool.data(), pool.size() * sizeof(int), cudaMemcpyHostToDevice));
  c->tabs.resize(ns->ops.size());
  for (size_t oi = 0; oi < ns->ops.size(); ++oi) {
    if (ns->ops[oi].kind != OP_CONV) continue;
    OpTables& t = c->tabs[oi];
    t.koff = c->table_pool + locs[oi].koff; t.kdhw = c->table_pool + locs[oi].kdhw; t.kci = c->table_pool + locs[oi].kci;
    t.koff_dx = c->table_pool + locs[oi].koff_dx; t.kdhw_dx = c->table_pool + locs[oi].kdhw_dx; t.kB_dx = c->table_pool + locs[oi].kB_dx;
  }
  BRL_CUDA(cudaMalloc(&c->site_off_dev, ns->site_off.size() * sizeof(long long)));
  BRL_CUDA(cudaMemcpy(c->site_off_dev, ns->site_off.data(), ns->site_off.size() * sizeof(long long), cudaMemcpyHostToDevice));
  for (size_t j = 0; j + 1 < ns->site_off.size(); ++j) c->max_site = std::max(c->max_site, (int)(ns->site_off[j + 1] - ns->site_off[j]));
  c->tc = tc_create(net);
  // dependency levels of the tape: an op is one level below the last producer of its input buffer
  c->op_level.assign(ns->ops.size(), 0);
  for (size_t oi = 0; oi < ns->ops.size(); ++oi) {
    int lvl = 0;
    for (size_t pj = 0; pj < oi; ++pj)
      if (ns->ops[pj].out_buf == ns->ops[oi].in.buf) lvl = std::max(lvl, c->op_level[pj] + 1);
    c->op_level[oi] = lvl;
    c->n_levels = std::max(c->n_levels, lvl + 1);
  }
  const char* single = getenv("BRL_SINGLE_STREAM");
  c->multi_stream = !(single && single[0] == '1');
  for (brl_ctx::Lane& ln : c->lanes) {
    for (int i = 0; i < 3; ++i) {
      BRL_CUDA(cudaStreamCreateWithFlags(&ln.side[i], cudaStreamNonBlocking));
      BRL_CUDA(cudaEventCreateWithFlags(&ln.ev_join[i], cudaEventDisableTiming));
    }
    BRL_CUDA(cudaEventCreateWithFlags(&ln.ev_fork, cudaEventDisableTiming));
    BRL_CUDA(cudaEventCreateWithFlags(&ln.ev_zero, cudaEventDisableTiming));
    BRL_CUDA(cudaStreamCreateWithFlags(&ln.zero, cudaStreamNonBlocking));
    for (int i = 0; i < 8; ++i) BRL_CUDA(cudaEventCreateWithFlags(&ln.ev_op[i], cudaEventDisableTiming));
  }
  BRL_CUDA(cudaStreamCreateWithFlags(&c->lane1_main, cudaStreamNonBlocking));
  c->lanes[1].main = c->lane1_main;
  BRL_CUDA(cudaEventCreateWithFlags(&c->ev_lane_fork, cudaEventDisableTiming));
  BRL_CUDA(cudaEventCreateWithFlags(&c->ev_lane_join, cudaEventDisableTiming));
  BRL_CUDA(cudaStreamCreateWithFlags(&c->cap, cudaStreamNonBlocking));
  BRL_CUDA(cudaStreamCreateWithFlags(&c->copy, cudaStreamNonBlocking));
  BRL_CUDA(cudaEventCreateWithFlags(&c->ev_copy_start, cudaEventDisableTiming));
  for (int i = 0; i < 8; ++i) BRL_CUDA(cudaEventCreateWithFlags(&c->ev_chunk[i], cudaEventDisableTiming));
  const char* nograph = getenv("BRL_NO_GRAPH");
  c->graph_enabled = !(nograph && nograph[0] == '1');
  *out = c;
  return BRL_OK;
}

int brl_destroy(brl_ctx* ctx) {
  if (!ctx) return BRL_OK;
  DeviceGuard dg(ctx->device);
  cudaFree(ctx->table_pool);
  cudaFree(ctx->site_off_dev);
  tc_destroy(ctx->tc);
  for (brl_ctx::Lane& ln : ctx->lanes) {
    for (int i = 0; i < 3; ++i) {
      if (ln.side[i]) cudaStreamDestroy(ln.side[i]);
      if (ln.ev_join[i]) cudaEventDestroy(ln.ev_join[i]);
    }
    if (ln.ev_fork) cudaEventDestroy(ln.ev_fork);
    if (ln.ev_zero) cudaEventDestroy(ln.ev_zero);
    if (ln.zero) cudaStreamDestroy(ln.zero);
    for (int i = 0; i < 8; ++i)
      if (ln.ev_op[i]) cudaEventDestroy(ln.ev_op[i]);
  }
  if (ctx->lane1_main) cudaStreamDestroy(ctx->lane1_main);
  if (ctx->ev_lane_fork) cudaEventDestroy(ctx->ev_lane_fork);
  if (ctx->ev_lane_join) cudaEventDestroy(ctx->ev_lane_join);
  for (auto& g : ctx->graphs)
    if (g.exec) cudaGraphExecDestroy(g.exec);
  if (ctx->cap) cudaStreamDestroy(ctx->cap);
  if (ctx->copy) cudaStreamDestroy(ctx->copy);
  if (ctx->ev_copy_start) cudaEventDestroy(ctx->ev_copy_start);
  for (int i = 0; i < 8; ++i)
    if (ctx->ev_chunk[i]) cudaEventDestroy(ctx->ev_chunk[i]);
  delete ctx;
  return BRL_OK;
}

int brl_tc_status(const brl_ctx* ctx) {
  if (!ctx) return -1;
  DeviceGuard dg(ctx->device);
  const int g = tc_gemm_status();  // TF32 per-layer kernels
  if (g != 0) return g;
  const int t = tt_status();  // level-fused training kernels
  if (t != 0) return t;
  return tc_status(ctx->tc);
}
int brl_gemm_status(void) { return tc_gemm_status(); }
int brl_set_gemm_backend(brl_ctx* ctx, int backend) {
  BRL_REQUIRE(ctx, "brl_set_gemm_backend: NULL context");
  BRL_REQUIRE(backend >= 0 && backend <= BRL_GEMM_TC_FUSED, "brl_set_gemm_backend: unknown back-end");
  ctx->gemm_backend = backend;
  return BRL_OK;
}
int brl_tc_timing(brl_ctx* ctx, int enable) {
  BRL_REQUIRE(ctx && tc_available(ctx->tc), "brl_tc_timing: tensor-core engine unavailable");
  tc_timing(ctx->tc, enable != 0);
  return BRL_OK;
}
int brl_tc_timing_read(brl_ctx* ctx, double* kernel_ms, int64_t* launches) {
  BRL_REQUIRE(ctx && kernel_ms && launches && tc_available(ctx->tc), "brl_tc_timing_read: bad argument");
  DeviceGuard dg(ctx->device);
  long long n[2] = {0, 0};
  tc_timing_read(ctx->tc, kernel_ms, n);
  launches[0] = n[0];
  launches[1] = n[1];
  return BRL_OK;
}
int brl_tt_trace(brl_ctx* ctx, int64_t* device_buf) {
  BRL_REQUIRE(ctx, "brl_tt_trace: NULL context");
  tt_trace(reinterpret_cast<long long*>(device_buf));
  return BRL_OK;
}
int brl_tc_trace(brl_ctx* ctx, int64_t* device_buf) {
  BRL_REQUIRE(ctx && tc_available(ctx->tc), "brl_tc_trace: tensor-core engine unavailable");
  tc_trace(ctx->tc, reinterpret_cast<long long*>(device_buf));
  return BRL_OK;
}

int brl_engine_available(const brl_ctx* ctx, int engine) {
  if (!ctx) return 0;
  if (engine == BRL_ENGINE_SIMT_FP32) return 1;
  if (engine == BRL_ENGINE_TC_FP16) return tc_available(ctx->tc) ? 1 : 0;
  return 0;
}

int64_t brl_workspace_bytes(const brl_ctx* ctx, int64_t B, int64_t S, int train, int engine) {
  if (!ctx || B <= 0 || S <= 0) return BRL_ERR_INVALID;
  const NetSpec& n = *ctx->net;
  Carve c(nullptr, 0);
  ActBufs ab;
  if (train == 5 || train == 6) {  // brl_elbo_train_steps / brl_hnn_train_steps: their buffers, then the step's workspace
    TrainBufs t;
    carve_train_steps(n, c, S, B, train == 5, t);
    const int64_t step = train == 5 ? (S == 1 ? brl_workspace_bytes(ctx, B, 2, 1, 0) : brl_workspace_bytes(ctx, B, S, 4, 0))
                                    : (S == 1 ? brl_workspace_bytes(ctx, B, 1, 1, 0) : brl_workspace_bytes(ctx, B, S, 3, 0));
    return (int64_t)c.used + step;
  }
  if (train == 7) {  // brl_elbo_val_steps: its buffers, then the larger of the ELBO step's workspace and the predictive's
    TrainBufs t;
    unsigned long long* key2;
    carve_val_steps(c, B, S, t, key2);
    Carve p(nullptr, 0);
    ValPredict v;
    const int64_t predict = (int64_t)carve_val_predict(ctx, p, B, S, engine, v);
    const int64_t elbo = brl_workspace_bytes(ctx, B, 2, 1, 0);  // two particle lanes: Engine.elbo_step's workspace for particles > 1
    return (int64_t)c.used + std::max(elbo, predict);
  }
  if (train == 3 || train == 4) {  // brl_hnn_step_ensemble / brl_elbo_step_ensemble over S members: the layout of their steps
    carve_forward(n, c, B, 1, ab);
    carve_train(n, c, B, ab);
    carve_tl(n, c, B, ab);
    carve_members(n, c, B, S, train == 4, ab);
    return (int64_t)c.used + 4096;
  }
  c.take<float>(4 * B);          // moment state
  c.take<float>(S * n.P);        // weight samples
  c.take<float>(S * 2 * (long long)n.layers.size());
  c.take<float>(S * B * 2);      // chunk outputs
  if (engine == BRL_ENGINE_TC_FP16) c.used += tc_workspace_bytes(ctx->tc, B, S);
  else carve_forward(n, c, B, S, ab);
  if (train == 1) carve_train(n, c, B, ab);
  ActBufs ab1;
  if (train == 1 && S >= 2) {  // second lane of brl_elbo_step: two particles side by side
    carve_forward(n, c, B, 1, ab1);
    carve_train(n, c, B, ab1);
  }
  if (train == 1) {  // fused Linear / Conv-D3 images of the lanes (brl_elbo_step / brl_hnn_step carve them last)
    carve_tl(n, c, B, ab);
    if (S >= 2) carve_tl(n, c, B, ab1);
  }
  if (train == 2)  // brl_forward in BRL_MODE_FLIPOUT with native signs: [S,B,Cin] + [S,B,Cout] per layer
    for (const LayerSpec& L : n.layers) { c.take<float>(S * B * L.cin); c.take<float>(S * B * L.cout); }
  return (int64_t)c.used + 4096;
}

int brl_sample_weights(brl_ctx* ctx, const float* mu, const float* sigma, int guide, int64_t S, const brl_noise* noise,
                       float* w_out, float* delta_out, void* workspace, size_t workspace_bytes, void* stream) {
  BRL_REQUIRE(ctx && mu && sigma && w_out && S > 0, "brl_sample_weights: NULL argument or S <= 0");
  DeviceGuard dg(ctx->device);
  const NetSpec& n = *ctx->net;
  cudaStream_t st = (cudaStream_t)stream;
  NoiseRef eps = nref(noise, noise ? noise->weight_eps : nullptr, KIND_WEIGHT_EPS, 0);
  if (guide == BRL_GUIDE_NORMAL) {
    launch_sample_normal(mu, sigma, n.P, S, eps, w_out, delta_out, st);
  } else if (guide == BRL_GUIDE_RADIAL) {
    const int ns = 2 * (int)n.layers.size();
    Carve c(workspace, workspace_bytes);
    float* norms = c.take<float>(S * ns);
    if (!workspace || !c.ok) return fail(BRL_ERR_WORKSPACE, "brl_sample_weights: workspace too small for radial norms");
    NoiseRef r = nref(noise, noise ? noise->radial_r : nullptr, KIND_RADIAL_R, 0);
    launch_sample_radial(mu, sigma, n.P, S, ctx->site_off_dev, ns, ctx->max_site, eps, r, norms, w_out, delta_out, st);
  } else {
    return fail(BRL_ERR_INVALID, "Guide unknown. Choose from 'normal', 'radial'.");
  }
  BRL_CUDA(cudaGetLastError());
  return BRL_OK;
}

static int resolve_signs(const brl_ctx* ctx, const brl_noise* nz, long long S, long long B, Carve& c,
                         std::vector<const float*>& sin_, std::vector<const float*>& sout_, cudaStream_t st) {
  const NetSpec& n = *ctx->net;
  sin_.assign(n.layers.size(), nullptr);
  sout_.assign(n.layers.size(), nullptr);
  for (size_t l = 0; l < n.layers.size(); ++l) {
    const LayerSpec& L = n.layers[l];
    if (nz && nz->flip_in[l]) sin_[l] = nz->flip_in[l];
    else {
      float* d = c.take<float>(S * B * L.cin);
      if (!c.ok) return fail(BRL_ERR_WORKSPACE, "workspace too small (flipout signs)");
      launch_gen_signs(d, S, B, L.cin, nref(nz, nullptr, KIND_FLIP_IN, (unsigned)l), st);
      sin_[l] = d;
    }
    if (nz && nz->flip_out[l]) sout_[l] = nz->flip_out[l];
    else {
      float* d = c.take<float>(S * B * L.cout);
      if (!c.ok) return fail(BRL_ERR_WORKSPACE, "workspace too small (flipout signs)");
      launch_gen_signs(d, S, B, L.cout, nref(nz, nullptr, KIND_FLIP_OUT, (unsigned)l), st);
      sout_[l] = d;
    }
  }
  return BRL_OK;
}

int brl_forward(brl_ctx* ctx, const float* x, int64_t B, int64_t S, int mode, const float* theta, const float* sigma,
                const float* wsamp, float p_dropout, const brl_noise* noise, float* out, int engine, void* workspace,
                size_t workspace_bytes, void* stream) {
  BRL_REQUIRE(ctx && x && out && workspace, "brl_forward: NULL argument");
  DeviceGuard dg(ctx->device);
  BRL_REQUIRE(B > 0 && S > 0 && B * 30 < (1ll << 31) / 512, "brl_forward: bad B or S");
  BRL_REQUIRE(mode >= BRL_MODE_DET && mode <= BRL_MODE_FLIPOUT, "brl_forward: unknown mode");
  BRL_REQUIRE(mode == BRL_MODE_WS || theta, "brl_forward: theta is NULL");
  BRL_REQUIRE(mode != BRL_MODE_LRT || sigma, "brl_forward: LRT needs sigma");
  BRL_REQUIRE((mode != BRL_MODE_WS && mode != BRL_MODE_FLIPOUT) || wsamp, "brl_forward: WS/FLIPOUT need wsamp [S,P]");
  BRL_REQUIRE(p_dropout >= 0.f && p_dropout < 1.f, "brl_forward: p_dropout must be in [0,1)");
  cudaStream_t st = (cudaStream_t)stream;
  const NetSpec& n = *ctx->net;
  if (engine == BRL_ENGINE_TC_FP16) {
    BRL_REQUIRE(mode == BRL_MODE_DET || mode == BRL_MODE_WS, "tensor-core engine supports DET / WS forward only");
    const char* err = tc_forward(ctx->tc, x, B, S, mode == BRL_MODE_WS ? wsamp : theta, mode == BRL_MODE_WS ? n.P : 0,
                                 p_dropout, noise, out, workspace, workspace_bytes, true, st);
    if (err) return fail(BRL_ERR_UNSUPPORTED, err);
    BRL_CUDA(cudaGetLastError());
    return BRL_OK;
  }
  BRL_REQUIRE(engine == BRL_ENGINE_SIMT_FP32, "unknown engine");
  Carve c(workspace, workspace_bytes);
  ActBufs ab;
  carve_forward(n, c, B, S, ab);
  if (!c.ok) return fail(BRL_ERR_WORKSPACE, "brl_forward: workspace too small");
  std::vector<const float*> sin_, sout_;
  if (mode == BRL_MODE_FLIPOUT) {
    int rc = resolve_signs(ctx, noise, S, B, c, sin_, sout_, st);
    if (rc) return rc;
  }
  FwdArgs fa{x, B, S, mode, theta, sigma, wsamp, p_dropout, noise, sin_.data(), sout_.data(), out, false};
  run_forward(ctx, ab, fa, st);
  BRL_CUDA(cudaGetLastError());
  return BRL_OK;
}

// largest chunk of S samples whose brl_predict_moments buffers fit `bytes` of workspace (at most 128 on the fused engine, whose
// per-sample footprint is 4.8 KB per window -- B = 10 000 x S = 100 is ONE pass over a 4.9 GB feature tensor: measured 4.60 /
// 4.50 / 4.46 ms per step for 25 / 50 / 100 samples per launch; 16 on the per-layer engines), then equal chunks; 0 when not
// even one sample fits
static long long sample_chunk(brl_ctx* ctx, long long B, long long S, int engine, size_t bytes) {
  static const int env_sc = getenv("BRL_TC_SC") ? atoi(getenv("BRL_TC_SC")) : 0;  // experiment knob
  long long Sc = std::min<long long>(S, engine == BRL_ENGINE_TC_FP16 ? (env_sc > 0 ? env_sc : 128) : 16);
  for (; Sc >= 1; --Sc)
    if ((size_t)brl_workspace_bytes(ctx, B, Sc, 0, engine) <= bytes) break;
  if (Sc >= 1) Sc = (S + (S + Sc - 1) / Sc - 1) / ((S + Sc - 1) / Sc);
  return std::max(Sc, 0ll);
}

int brl_predict_moments(brl_ctx* ctx, const float* x, int64_t B, int64_t S, int guide, const float* mu,
                        const float* sigma, float p_dropout, const brl_noise* noise, float* pred, float* std,
                        float* ep_var, float* al_var, int engine, void* workspace, size_t workspace_bytes, void* stream) {
  BRL_REQUIRE(ctx && x && mu && pred && std && workspace, "brl_predict_moments: NULL argument");
  DeviceGuard dg(ctx->device);
  BRL_REQUIRE(B > 0 && S > 0 && B * 30 < (1ll << 31) / 512, "brl_predict_moments: bad B or S");
  BRL_REQUIRE(guide < 0 || sigma, "brl_predict_moments: sigma is NULL");
  BRL_REQUIRE(guide <= BRL_GUIDE_RADIAL, "Guide unknown. Choose from 'normal', 'radial'.");
  cudaStream_t st = (cudaStream_t)stream;
  const NetSpec& n = *ctx->net;
  const int nsites = 2 * (int)n.layers.size();
  const long long Sc = sample_chunk(ctx, B, S, engine, workspace_bytes);
  if (Sc < 1) return fail(BRL_ERR_WORKSPACE, "brl_predict_moments: workspace too small for one MC sample; need " +
                                                 std::to_string(brl_workspace_bytes(ctx, B, 1, 0, engine)) + " bytes");
  Carve c(workspace, workspace_bytes);
  float* state = c.take<float>(4 * B);
  float* wsamp = c.take<float>(Sc * n.P);
  float* norms = c.take<float>(Sc * nsites);
  float* outc = c.take<float>(Sc * B * 2);
  ActBufs ab;
  void* tc_ws = nullptr;
  size_t tc_bytes = 0;
  if (engine == BRL_ENGINE_TC_FP16) {
    tc_bytes = tc_workspace_bytes(ctx->tc, B, Sc);
    tc_ws = c.take<char>((long long)tc_bytes);
  } else {
    carve_forward(n, c, B, Sc, ab);
  }
  if (!c.ok) return fail(BRL_ERR_WORKSPACE, "brl_predict_moments: workspace carve failed");
  for (long long s0 = 0; s0 < S; s0 += Sc) {
    const long long sc = std::min(Sc, S - s0);
    brl_noise nz = noise_at_sample(n, noise, s0, B);
    const float* w = mu;
    int mode = BRL_MODE_DET;
    if (guide >= 0) {
      NoiseRef eps = nref(&nz, nz.weight_eps, KIND_WEIGHT_EPS, 0);
      if (guide == BRL_GUIDE_NORMAL) launch_sample_normal(mu, sigma, n.P, sc, eps, wsamp, nullptr, st);
      else launch_sample_radial(mu, sigma, n.P, sc, ctx->site_off_dev, nsites, ctx->max_site, eps,
                                nref(&nz, nz.radial_r, KIND_RADIAL_R, 0), norms, wsamp, nullptr, st);
      w = wsamp;
      mode = BRL_MODE_WS;
    }
    if (engine == BRL_ENGINE_TC_FP16) {
      const char* err = tc_forward(ctx->tc, x, B, sc, w, mode == BRL_MODE_WS ? n.P : 0, p_dropout, &nz, outc, tc_ws, tc_bytes, s0 == 0, st);
      if (err) return fail(BRL_ERR_UNSUPPORTED, err);
    } else {
      FwdArgs fa{x, B, sc, mode, w, nullptr, w, p_dropout, &nz, nullptr, nullptr, outc, false};
      run_forward(ctx, ab, fa, st);
    }
    launch_moments_update(outc, sc, B, state, s0 == 0, st);
  }
  launch_moments_final(state, B, pred, std, ep_var, al_var, st);
  BRL_CUDA(cudaGetLastError());
  return BRL_OK;
}

// M members' moments over one batch.  The M S draws form ONE member-major sample axis j = m S + s (MC-sample index sample0 + j,
// injected noise row j), cut into chunks as brl_predict_moments cuts S.  On the tensor-core engine each chunk is one sampler
// launch (draw j from member j / S), one pack launch (one image per draw, or per member for MC-dropout / deterministic
// members), the engine's kernels and one member-routed Welford update; every member's samples go through the same arithmetic
// as in its own call, whatever chunk they fall in.  Elsewhere the members run one after another on brl_predict_moments.
int brl_predict_moments_ensemble(brl_ctx* ctx, const float* x, int64_t M, int64_t B, int64_t S, int guide, const float* mu,
                                 const float* sigma, float p_dropout, const brl_noise* noise, float* out, int engine, void* workspace,
                                 size_t workspace_bytes, void* stream) {
  BRL_REQUIRE(ctx && x && mu && out && workspace, "brl_predict_moments_ensemble: NULL argument");
  DeviceGuard dg(ctx->device);
  BRL_REQUIRE(M > 0 && M < (1 << 16) && B > 0 && S > 0 && B * 30 < (1ll << 31) / 512 && S < (1ll << 31) / M,
              "brl_predict_moments_ensemble: bad M, B or S");
  BRL_REQUIRE(p_dropout >= 0.f && p_dropout < 1.f, "brl_predict_moments_ensemble: p_dropout must be in [0,1)");
  BRL_REQUIRE(guide < 0 || sigma, "brl_predict_moments_ensemble: sigma is NULL");
  BRL_REQUIRE(guide <= BRL_GUIDE_RADIAL, "Guide unknown. Choose from 'normal', 'radial'.");
  cudaStream_t st = (cudaStream_t)stream;
  const NetSpec& n = *ctx->net;
  const size_t state_bytes = ((size_t)(M * 4 * B) * sizeof(float) + 255) & ~(size_t)255;  // Welford state [M,4,B]
  const size_t need = (size_t)brl_workspace_bytes(ctx, B, 1, 0, engine) + state_bytes;
  if (workspace_bytes < need)
    return fail(BRL_ERR_WORKSPACE, "brl_predict_moments_ensemble: workspace too small; need " + std::to_string(need) + " bytes");
  brl_noise base;
  memset(&base, 0, sizeof(base));
  if (noise) base = *noise;
  // the Linear and Conv-D3 tensor-core engines have no dropout path: their members run (and fail) as single calls
  const bool batched = engine == BRL_ENGINE_TC_FP16 && tc_available(ctx->tc) && (p_dropout == 0.f || n.id == BRL_NET_INCEPTION);
  if (!batched) {
    for (int64_t m = 0; m < M; ++m) {
      const brl_noise nm = noise_at_sample(n, &base, m * S, B);  // MC-sample index sample0 + m S, injected rows of member m
      const int rc = brl_predict_moments(ctx, x, B, S, guide, mu + m * n.P, guide >= 0 ? sigma + m * n.P : nullptr, p_dropout, &nm,
                                         out + m * B, out + (M + m) * B, out + (2 * M + m) * B, out + (3 * M + m) * B, engine,
                                         workspace, workspace_bytes, stream);
      if (rc != BRL_OK) return rc;
    }
    return BRL_OK;
  }
  const long long T = M * S;
  const long long Sc = sample_chunk(ctx, B, T, engine, workspace_bytes - state_bytes);
  const int nsites = 2 * (int)n.layers.size();
  Carve c(workspace, workspace_bytes);
  float* state = c.take<float>(M * 4 * B);
  float* wsamp = c.take<float>(Sc * n.P);
  float* norms = c.take<float>(Sc * nsites);
  float* outc = c.take<float>(Sc * B * 2);
  const size_t tc_bytes = tc_workspace_bytes(ctx->tc, B, Sc);
  void* tc_ws = c.take<char>((long long)tc_bytes);
  if (Sc < 1 || !c.ok) return fail(BRL_ERR_WORKSPACE, "brl_predict_moments_ensemble: workspace carve failed");
  for (long long j0 = 0; j0 < T; j0 += Sc) {
    const long long sc = std::min(Sc, T - j0), m0 = j0 / S, phase = j0 - m0 * S;  // the chunk starts `phase` samples into member m0
    brl_noise nz = noise_at_sample(n, &base, j0, B);
    const char* err;
    if (guide >= 0) {
      NoiseRef eps = nref(&nz, nz.weight_eps, KIND_WEIGHT_EPS, 0);
      if (guide == BRL_GUIDE_NORMAL)
        launch_sample_normal(mu + m0 * n.P, sigma + m0 * n.P, n.P, sc, eps, wsamp, nullptr, st, n.P, 1, (int)S, (int)phase);
      else
        launch_sample_radial(mu + m0 * n.P, sigma + m0 * n.P, n.P, sc, ctx->site_off_dev, nsites, ctx->max_site, eps,
                             nref(&nz, nz.radial_r, KIND_RADIAL_R, 0), norms, wsamp, nullptr, st, n.P, 1, (int)S, (int)phase);
      err = tc_forward(ctx->tc, x, B, sc, wsamp, n.P, p_dropout, &nz, outc, tc_ws, tc_bytes, j0 == 0, st);
    } else {  // one image per member: draw j reads image j / S of the members from m0 on
      err = tc_forward(ctx->tc, x, B, sc, mu + m0 * n.P, n.P, p_dropout, &nz, outc, tc_ws, tc_bytes, j0 == 0, st, nullptr, (int)S,
                       (int)phase);
    }
    if (err) return fail(BRL_ERR_UNSUPPORTED, err);
    launch_moments_update_members(outc, j0, sc, S, B, state, st);
  }
  launch_moments_final_members(state, M, B, out, st);
  BRL_CUDA(cudaGetLastError());
  return BRL_OK;
}

// ---- host-buffer variant of brl_predict_moments --------------------------------------------------------------------
// Window chunks: NW = 2 for large batches on the fused engine (measured, B = 10 000 x S = 100, ms per step end to end:
// NW = 1 4.99, 2 4.87, 3 5.05, 4 4.97, 6 5.17, 8 5.36 -- every further chunk costs ~0.1 ms of kernel ramp-up / drain, more than
// the copy it hides), rounded to 128 windows.  Per chunk, MC samples run in sub-chunks that fit the feature buffer.  The fp16 weight images of ALL S samples are packed once, up front (while the
// first chunk is still in flight), and shared by the chunks.
struct HostPlan {
  long long B0, Bc, n_chunks, Sc, Sw;  // windows of the first / of every later chunk, chunks, samples per feature-buffer pass,
                                       // samples per sampler pass.  Buffers are sized for Bc >= B0.
  void range(long long B, long long ci, long long& w0, long long& bc) const {
    w0 = ci == 0 ? 0 : B0 + (ci - 1) * Bc;
    bc = ci == 0 ? B0 : std::min(Bc, B - w0);
  }
};
static bool noise_is_native(const brl_noise* nz);
static HostPlan host_plan(const brl_ctx* ctx, long long B, long long S, int engine, bool native) {
  HostPlan p;
  static const int env_nw = getenv("BRL_HOST_NW") ? atoi(getenv("BRL_HOST_NW")) : 0;  // experiment knob
  p.n_chunks = (engine == BRL_ENGINE_TC_FP16 && native && B >= 4096) ? (env_nw > 0 ? std::min(env_nw, 8) : 2) : 1;
  static const int env_first = getenv("BRL_HOST_FIRST_PCT") ? atoi(getenv("BRL_HOST_FIRST_PCT")) : 30;  // experiment knob
  if (p.n_chunks == 1) {
    p.B0 = p.Bc = B;
  } else {  // a smaller first chunk exposes less of its copy; the later chunks share the rest evenly
    p.B0 = std::min(B, std::max<long long>(128, (B * env_first / 100 + 127) / 128 * 128));
    p.Bc = std::max(p.B0, (((B - p.B0) + p.n_chunks - 2) / (p.n_chunks - 1) + 127) / 128 * 128);
    p.n_chunks = 1 + (B - p.B0 + p.Bc - 1) / p.Bc;
  }
  p.Sw = std::min<long long>(S, 16);
  p.Sc = S;
  if (engine == BRL_ENGINE_TC_FP16)
    while (p.Sc > 1 && tc_workspace_bytes(ctx->tc, p.Bc, p.Sc) > ((size_t)4 << 30)) p.Sc = (p.Sc + 1) / 2;  // feature buffer <= 4 GB
  return p;
}
struct HostCarve {
  float *x_dev, *res, *state, *wsamp, *norms, *outc;
  unsigned char* images;
  void* tc_ws;
  size_t tc_bytes;
};
static bool host_carve(const brl_ctx* ctx, Carve& c, long long B, long long S, int guide, const HostPlan& pl, HostCarve& h) {
  const NetSpec& n = *ctx->net;
  h.x_dev = c.take<float>(B * 540);
  h.res = c.take<float>(4 * B);
  h.state = c.take<float>(4 * pl.Bc);
  h.wsamp = c.take<float>(pl.Sw * n.P);
  h.norms = c.take<float>(pl.Sw * 2 * (long long)n.layers.size());
  h.outc = c.take<float>(pl.Sc * pl.Bc * 2);
  h.images = c.take<unsigned char>((guide >= 0 ? S : 1) * (long long)tc_weight_image_bytes());
  h.tc_bytes = tc_workspace_bytes(ctx->tc, pl.Bc, pl.Sc);
  h.tc_ws = c.take<char>((long long)h.tc_bytes);
  return c.ok;
}

int64_t brl_workspace_bytes_host(const brl_ctx* ctx, int64_t B, int64_t S, int engine) {
  if (!ctx || B <= 0 || S <= 0) return BRL_ERR_INVALID;
  if (engine != BRL_ENGINE_TC_FP16 || !tc_host_pipeline(ctx->tc)) {
    const bool tc = engine == BRL_ENGINE_TC_FP16 && tc_available(ctx->tc);  // (Linear net: one copy, then the device entry point)
    return brl_workspace_bytes(ctx, B, std::min<int64_t>(S, tc ? 128 : 16), 0, tc ? BRL_ENGINE_TC_FP16 : BRL_ENGINE_SIMT_FP32) +
           (B * 540 + 4 * B) * (int64_t)sizeof(float) + 1024;
  }
  size_t need = 0;
  for (int native = 0; native < 2; ++native) {  // injected noise runs as ONE window chunk (larger per-chunk buffers): size for both
    Carve c(nullptr, 0);
    HostCarve h;
    host_carve(ctx, c, B, S, 0, host_plan(ctx, B, S, engine, native != 0), h);
    need = std::max(need, c.used);
  }
  return (int64_t)need + 4096;
}

int brl_predict_moments_host(brl_ctx* ctx, const float* x_host, int64_t B, int64_t S, int guide, const float* mu,
                             const float* sigma, float p_dropout, const brl_noise* noise, float* out_host, int engine,
                             void* workspace, size_t workspace_bytes, void* stream) {
  BRL_REQUIRE(ctx && x_host && mu && out_host && workspace, "brl_predict_moments_host: NULL argument");
  DeviceGuard dg(ctx->device);
  BRL_REQUIRE(B > 0 && S > 0 && B * 30 < (1ll << 31) / 512, "brl_predict_moments_host: bad B or S");
  BRL_REQUIRE(guide < 0 || sigma, "brl_predict_moments_host: sigma is NULL");
  BRL_REQUIRE(guide <= BRL_GUIDE_RADIAL, "Guide unknown. Choose from 'normal', 'radial'.");
  cudaStream_t st = (cudaStream_t)stream;
  const NetSpec& n = *ctx->net;
  const size_t xbytes = sizeof(float) * (size_t)B * 540;
  if (engine != BRL_ENGINE_TC_FP16 || !tc_host_pipeline(ctx->tc)) {
    // per-layer engine (or the Linear net's tensor-core engine): one copy, then the device entry point on the rest of the workspace
    const int dev_engine = (engine == BRL_ENGINE_TC_FP16 && tc_available(ctx->tc)) ? BRL_ENGINE_TC_FP16 : BRL_ENGINE_SIMT_FP32;
    Carve c(workspace, workspace_bytes);
    float* x_dev = c.take<float>(B * 540);
    float* res = c.take<float>(4 * B);
    if (!c.ok) return fail(BRL_ERR_WORKSPACE, "brl_predict_moments_host: workspace too small");
    BRL_CUDA(cudaMemcpyAsync(x_dev, x_host, xbytes, cudaMemcpyHostToDevice, st));
    int rc = brl_predict_moments(ctx, x_dev, B, S, guide, mu, sigma, p_dropout, noise, res, res + B, res + 2 * B, res + 3 * B,
                                 dev_engine, (char*)workspace + c.used, workspace_bytes - c.used, stream);
    if (rc) return rc;
    BRL_CUDA(cudaMemcpyAsync(out_host, res, sizeof(float) * 4 * B, cudaMemcpyDeviceToHost, st));
    return BRL_OK;
  }
  const HostPlan pl = host_plan(ctx, B, S, engine, noise_is_native(noise));
  BRL_REQUIRE(pl.n_chunks <= 8, "brl_predict_moments_host: too many window chunks");
  Carve c(workspace, workspace_bytes);
  HostCarve h;
  if (!host_carve(ctx, c, B, S, guide, pl, h))
    return fail(BRL_ERR_WORKSPACE, "brl_predict_moments_host: workspace too small; need " +
                                       std::to_string(brl_workspace_bytes_host(ctx, B, S, engine)) + " bytes");
  // ---- copies: one per window chunk, on the copy stream, behind whatever still uses the workspace on `st`
  BRL_CUDA(cudaEventRecord(ctx->ev_copy_start, st));
  BRL_CUDA(cudaStreamWaitEvent(ctx->copy, ctx->ev_copy_start, 0));
  for (long long ci = 0; ci < pl.n_chunks; ++ci) {
    long long w0, bc;
    pl.range(B, ci, w0, bc);
    BRL_CUDA(cudaMemcpyAsync(h.x_dev + w0 * 540, x_host + w0 * 540, sizeof(float) * bc * 540, cudaMemcpyHostToDevice, ctx->copy));
    BRL_CUDA(cudaEventRecord(ctx->ev_chunk[ci], ctx->copy));
  }
  // ---- weight images of all MC samples (no dependence on x: runs underneath the first copy)
  const int nsites = 2 * (int)n.layers.size();
  if (guide >= 0) {
    for (long long s0 = 0; s0 < S; s0 += pl.Sw) {
      const long long sw = std::min(pl.Sw, S - s0);
      brl_noise nz = noise_at_sample(n, noise, s0, B);
      NoiseRef eps = nref(&nz, nz.weight_eps, KIND_WEIGHT_EPS, 0);
      if (guide == BRL_GUIDE_NORMAL) launch_sample_normal(mu, sigma, n.P, sw, eps, h.wsamp, nullptr, st);
      else launch_sample_radial(mu, sigma, n.P, sw, ctx->site_off_dev, nsites, ctx->max_site, eps,
                                nref(&nz, nz.radial_r, KIND_RADIAL_R, 0), h.norms, h.wsamp, nullptr, st);
      const char* err = tc_pack_weights(ctx->tc, h.wsamp, n.P, sw, h.images + s0 * (long long)tc_weight_image_bytes(), p_dropout, st);
      if (err) return fail(BRL_ERR_UNSUPPORTED, err);
    }
  } else {
    const char* err = tc_pack_weights(ctx->tc, mu, 0, 1, h.images, p_dropout, st);
    if (err) return fail(BRL_ERR_UNSUPPORTED, err);
  }
  // ---- chunks of windows x sub-chunks of samples
  for (long long ci = 0; ci < pl.n_chunks; ++ci) {
    long long w0, bc;
    pl.range(B, ci, w0, bc);
    BRL_CUDA(cudaStreamWaitEvent(st, ctx->ev_chunk[ci], 0));
    for (long long s0 = 0; s0 < S; s0 += pl.Sc) {
      const long long sc = std::min(pl.Sc, S - s0);
      brl_noise nz = noise_at_sample(n, noise, s0, B);
      nz.window0 += w0;
      const unsigned char* img = h.images + (guide >= 0 ? s0 * (long long)tc_weight_image_bytes() : 0);
      const char* err = tc_forward(ctx->tc, h.x_dev + w0 * 540, bc, sc, nullptr, guide >= 0 ? n.P : 0, p_dropout, &nz, h.outc,
                                   h.tc_ws, h.tc_bytes, s0 == 0, st, img);
      if (err) return fail(BRL_ERR_UNSUPPORTED, err);
      launch_moments_update(h.outc, sc, bc, h.state, s0 == 0, st);
    }
    launch_moments_final(h.state, bc, h.res + w0, h.res + B + w0, h.res + 2 * B + w0, h.res + 3 * B + w0, st);
  }
  BRL_CUDA(cudaMemcpyAsync(out_host, h.res, sizeof(float) * 4 * B, cudaMemcpyDeviceToHost, st));
  BRL_CUDA(cudaGetLastError());
  return BRL_OK;
}

int brl_moments(const float* out, int64_t S, int64_t B, float* pred, float* std, float* ep_var, float* al_var, void* stream) {
  BRL_REQUIRE(out && pred && std && S > 0 && B > 0, "brl_moments: bad argument");
  BRL_REQUIRE(ep_var && al_var, "brl_moments: ep_var / al_var must be given");
  cudaStream_t st = (cudaStream_t)stream;
  launch_moments_direct(out, S, B, pred, std, ep_var, al_var, st);
  BRL_CUDA(cudaGetLastError());
  return BRL_OK;
}

int brl_aggregate_predictions(const float* out, int64_t S, int64_t B, float* agg, void* stream) {
  BRL_REQUIRE(out && agg && S > 0 && B > 0, "brl_aggregate_predictions: bad argument");
  launch_aggregate(out, S, B, agg, (cudaStream_t)stream);
  BRL_CUDA(cudaGetLastError());
  return BRL_OK;
}

// ---- level-fused tcgen05 training kernels (BRL_GEMM_TC_FUSED) of the three nets, shared by the ELBO and HNN steps: layers 0..L-1
// on the tensor pipe, the rest of the net (the epilogue of fc layer `fc` if there is one, the head, the likelihood and their
// backward) in one tt_tail launch over the `width` hidden units in front of the head (always the last layer)
struct FusedNet { int L, fc, width; };
static FusedNet fused_net(const NetSpec& n) {
  if (n.id == BRL_NET_INCEPTION) return {TT_LAYERS, TT_LAYERS, 64};  // ten convs, fc layer 10
  if (n.id == BRL_NET_LINEAR) return {4, 3, 32};                      // four hidden layers, the tail runs layer 3's epilogue
  return {3, -1, 320};                                                 // Conv-D3: three convs, the head reads the pooled features
}

// M members of a step in ONE chain of launches on the fused kernels: this net's images carved for M members (more than one: the
// Inception net only) and, for the Inception net, the fc layer's partial sums within the split-K scratch (B <= 4736).  Every mode
// the ELBO step (LRT / Flipout / WS) and the HNN step (DET) accept runs on them.
static bool fused_ok(const brl_ctx* ctx, const ActBufs& ab, long long M, long long B) {
  return ctx->gemm_backend == BRL_GEMM_TC_FUSED && ab.fused && M <= ab.fused_members &&
         (ctx->net->id != BRL_NET_INCEPTION || 2 * B * 64 <= SPLITK_SCRATCH_FLOATS);
}

static float keep_prob(const LayerSpec& L, float p_dropout) {
  return (p_dropout > 0.f && L.drop_factor > 0.f) ? 1.0f - p_dropout * L.drop_factor : 1.0f;
}

// the fused kernels' view of one particle lane of the step `a` describes: LRT eps (ELBO) or dropout sites (mode DET: the HNN step)
// and the sign tensors of layers 0..L-1, the members' strides (read against blockIdx.z only, so inert at M = 1)
static TtStep fused_step(const brl_ctx* ctx, const ActBufs& ab, const FwdArgs& a, long long M, float* g0, float* g1, int particles) {
  const NetSpec& n = *ctx->net;
  const FusedNet f = fused_net(n);
  const brl_noise& nz = *a.noise;
  auto sin_ = [&](int ly) { return a.sgn_in ? a.sgn_in[ly] : nullptr; };
  TtStep ts{};
  // weight-sampling ELBO (radial guide / no fit context): ONE contraction with the particle's weight draw
  ts.x = a.x; ts.B = a.B; ts.mode = a.mode; ts.mu = a.mode == BRL_MODE_WS ? a.wsamp : a.theta; ts.sigma = a.sigma; ts.wsamp = a.wsamp;
  for (int ly = 0; ly < f.L; ++ly) {
    if (a.mode == BRL_MODE_DET) ts.drop[ly] = nref(&nz, nz.drop_mask[ly], KIND_DROPOUT, (unsigned)ly);
    else ts.eps[ly] = nref(&nz, nz.lrt_eps[ly], KIND_LRT_EPS, (unsigned)ly);
    ts.keep[ly] = keep_prob(n.layers[ly], a.p_dropout);
    ts.sgn_in[ly] = sin_(ly); ts.sgn_out[ly] = a.sgn_out ? a.sgn_out[ly] : nullptr;
    ts.w_off[ly] = n.layers[ly].w_off; ts.b_off[ly] = n.layers[ly].b_off;
  }
  (f.L < TT_LAYERS ? ts.sgn_in[f.L] : ts.sgn_fc_in) = sin_(f.L);  // s_in of the first layer behind the tensor pipe
  if (f.fc >= 0) { ts.w_off_fc = n.layers[f.fc].w_off; ts.b_off_fc = n.layers[f.fc].b_off; }
  ts.g0 = g0; ts.g1 = g1;
  ts.members = (int)M; ts.P = n.P; ts.lane_stride = ab.fused_stride;
  ts.noise_stride = particles; ts.sign_stride = nz.flip_in[0] ? particles : 1;
  return ts;
}

static void fused_forward(const brl_ctx* ctx, const ActBufs& ab, const TtStep& ts, cudaStream_t st, const TtSide& sd) {
  if (ctx->net->id == BRL_NET_INCEPTION) {
    tt_forward(ab.tt, ts, st, sd);
    tt_fc_forward(ab.tt, ts, ab.part[0], st);
  } else if (ctx->net->id == BRL_NET_LINEAR) {
    tl_forward(ab.tl, ts, st, sd);
  } else {
    tc3_forward(ab.tc3, ts, st, sd);
  }
}

// the tail: the ELBO likelihood (gscale = c_nll / particles, acc [M][4]) or in mode DET the HNN loss (acc [M][2]) of `a`'s lane
static void fused_tail(const brl_ctx* ctx, const ActBufs& ab, const TtStep& ts, const FwdArgs& a, const float* y, float gscale,
                       int compute_grads, double* acc, cudaStream_t st) {
  const NetSpec& n = *ctx->net;
  const FusedNet f = fused_net(n);
  const brl_noise& nz = *a.noise;
  const int hd = (int)n.layers.size() - 1, fc_op = (int)n.ops.size() - 2;
  TtTail tl{};
  tl.part = n.id == BRL_NET_INCEPTION ? ab.part[0] : n.id == BRL_NET_LINEAR ? ab.tl.part : ab.tc3.feat;
  tl.width = f.width; tl.y = y; tl.gscale = gscale; tl.compute_grads = compute_grads; tl.acc = acc; tl.out = a.out;
  tl.dpre = f.fc >= 0 ? ab.dpre[fc_op] : ab.tc3.dfeat;
  tl.dsec = f.fc >= 0 ? ab.dsec[fc_op] : nullptr;
  tl.hw_off = n.layers[hd].w_off; tl.hb_off = n.layers[hd].b_off;
  if (a.mode == BRL_MODE_DET) {
    tl.loss_kind = 1;
    if (f.fc >= 0) {
      tl.keep_fc = keep_prob(n.layers[f.fc], a.p_dropout);
      tl.drop_fc = nref(&nz, nz.drop_mask[f.fc], KIND_DROPOUT, (unsigned)f.fc);
    }
  } else {
    if (f.fc >= 0) { tl.eps_fc = nref(&nz, nz.lrt_eps[f.fc], KIND_LRT_EPS, (unsigned)f.fc); tl.sout_fc = a.sgn_out[f.fc]; }
    tl.eps_head = nref(&nz, nz.lrt_eps[hd], KIND_LRT_EPS, (unsigned)hd);
    tl.sin_head = a.sgn_in[hd]; tl.sout_head = a.sgn_out[hd];
    tl.acc_stride = 4;
  }
  tt_tail(ts, tl, st);
}

static void fused_backward(const brl_ctx* ctx, const ActBufs& ab, const TtStep& ts, cudaStream_t st, const TtSide& sd) {
  const int fc_op = (int)ctx->net->ops.size() - 2;
  if (ctx->net->id == BRL_NET_INCEPTION) {
    tt_fc_backward(ab.tt, ts, ab.dpre[fc_op], ab.dsec[fc_op], st, sd);
    tt_backward(ab.tt, ts, st, sd);
  } else if (ctx->net->id == BRL_NET_LINEAR) {
    tl_backward(ab.tl, ts, ab.dpre.data(), ab.dsec.data(), st, sd);
  } else {
    tc3_backward(ab.tc3, ts, st, sd);
  }
}

// injected Flipout signs of the member-batched kernels: member m's tensors start `particles` rows [B, C] after member m - 1's,
// the signs generated in the workspace one row after; with several particles the kernels take one stride for all layers
static bool signs_one_stride(const NetSpec& n, const brl_noise* nz, int particles) {
  if (!nz || particles == 1) return true;
  int injected = 0;
  for (size_t l = 0; l < n.layers.size(); ++l) injected += (nz->flip_in[l] != nullptr) + (nz->flip_out[l] != nullptr);
  return injected == 0 || injected == 2 * (int)n.layers.size();
}

// the launches of one ELBO step of M members (every pointer final; M > 1 only where fused_ok holds); captured as is by the
// graph path of elbo_step.
// lanes[0] always exists and owns the shared accumulators; with a second buffer set (lanes[1]) two particles run side by
// side: lane 0 on `st`, lane 1 on the context's own stream, forked / joined with events.  The gradient finalisation of the
// particles (first one writes, the others accumulate) stays in particle order on `st`.  M > 1 members share every launch of one
// lane (member m on blockIdx.z of the fused kernels, on blockIdx.y of the sampler / sign / finalisation kernels), particle after
// particle; their accumulators are [M][4].
static int elbo_body(brl_ctx* ctx, const ActBufs* const* lanes, int n_lanes, const float* x, const float* y, int64_t M, int64_t B,
                     const float* mu, const float* sigma, int mode, int guide, int particles, float prior_loc, float prior_scale,
                     int64_t dataset_size, const brl_noise* noise, int compute_grads, double* scalars, float* grad_mu,
                     float* grad_sigma, float* grad_log_sigma, float* out, cudaStream_t st) {
  const NetSpec& n = *ctx->net;
  const ActBufs& ab0 = *lanes[0];
  const double cc = 1.0 / ((double)dataset_size * 30.0 * 18.0);
  const double c_nll = cc * (double)dataset_size / (double)B;
  BRL_CUDA(cudaMemsetAsync(ab0.acc, 0, std::max<int64_t>(8, 4 * M) * sizeof(double), st));
  const int nsites = 2 * (int)n.layers.size();
  if (!ctx->multi_stream || M > 1) n_lanes = 1;
  for (int p0 = 0; p0 < particles; p0 += n_lanes) {
    const int nl = std::min(n_lanes, particles - p0);
    if (nl > 1) {
      BRL_CUDA(cudaEventRecord(ctx->ev_lane_fork, st));
      BRL_CUDA(cudaStreamWaitEvent(ctx->lane1_main, ctx->ev_lane_fork, 0));
    }
    for (int l = 0; l < nl; ++l) {
      const int pt = p0 + l;
      const ActBufs& ab = *lanes[l];
      cudaStream_t ls = l == 0 ? st : ctx->lane1_main;
      brl_noise nz = noise_at_sample(n, noise, pt, B);
      const bool need_w = mode != BRL_MODE_LRT;
      if (need_w) {
        NoiseRef eps = nref(&nz, nz.weight_eps, KIND_WEIGHT_EPS, 0);
        // one draw per member: member m's posterior, MC-sample index sample0 + m particles + pt
        if (guide == BRL_GUIDE_NORMAL) launch_sample_normal(mu, sigma, n.P, M, eps, ab.wsamp, ab.delta, ls, n.P, particles);
        else launch_sample_radial(mu, sigma, n.P, M, ctx->site_off_dev, nsites, ctx->max_site, eps,
                                  nref(&nz, nz.radial_r, KIND_RADIAL_R, 0), ab.norms, ab.wsamp, ab.delta, ls, n.P, particles);
      }
      std::vector<const float*> sin_(n.layers.size(), nullptr), sout_(n.layers.size(), nullptr);
      if (mode == BRL_MODE_FLIPOUT) {  // native sign tensors of all layers: one launch per particle
        SignJobs jobs;
        jobs.n = 0;
        jobs.start[0] = 0;
        auto add = [&](float* dst, int C, unsigned kind, unsigned site) {
          jobs.dst[jobs.n] = dst; jobs.C[jobs.n] = C; jobs.kind[jobs.n] = kind; jobs.site[jobs.n] = site;
          jobs.start[jobs.n + 1] = jobs.start[jobs.n] + B * ((C + 3) / 4);  // work items: one Philox block = four channels
          ++jobs.n;
        };
        for (size_t ly = 0; ly < n.layers.size(); ++ly) {
          if (nz.flip_in[ly]) sin_[ly] = nz.flip_in[ly];
          else { add(ab.sgn_in[ly], n.layers[ly].cin, KIND_FLIP_IN, (unsigned)ly); sin_[ly] = ab.sgn_in[ly]; }
          if (nz.flip_out[ly]) sout_[ly] = nz.flip_out[ly];
          else { add(ab.sgn_out[ly], n.layers[ly].cout, KIND_FLIP_OUT, (unsigned)ly); sout_[ly] = ab.sgn_out[ly]; }
        }
        if (jobs.n) launch_gen_signs_multi(jobs, B, nref(&nz, nullptr, 0, 0), ls, (int)M, particles);
      }
      float* outp = out + (long long)pt * B * 2;
      const brl_ctx::Lane& ln = ctx->lanes[l];
      const TtSide sd{ln.side[0], ln.ev_fork, ln.ev_join[0]};
      const bool fused = fused_ok(ctx, ab, M, B);
      if (compute_grads) {  // a dozen memsets: on a side stream underneath the forward pass, joined before the NLL
        cudaStream_t zs = ctx->multi_stream ? ln.zero : ls;
        if (zs != ls) {
          BRL_CUDA(cudaEventRecord(ln.ev_zero, ls));
          BRL_CUDA(cudaStreamWaitEvent(zs, ln.ev_zero, 0));
        }
        if (!fused) {  // the fused back-end keeps its gradients in bf16 images that are written, not accumulated
          int rc = zero_grads(n, ab, B, zs);
          if (rc) return rc;
        }
        BRL_CUDA(cudaMemsetAsync(ab.g0, 0, sizeof(float) * M * n.P, zs));
        BRL_CUDA(cudaMemsetAsync(ab.g1, 0, sizeof(float) * M * n.P, zs));
        if (zs != ls) BRL_CUDA(cudaEventRecord(ln.ev_zero, zs));
      }
      FwdArgs fa{x, B, 1, mode, mu, sigma, ab.wsamp, 0.f, &nz, sin_.data(), sout_.data(), outp, compute_grads != 0};
      const TtStep ts = fused ? fused_step(ctx, ab, fa, M, ab.g0, ab.g1, particles) : TtStep{};
      if (fused) fused_forward(ctx, ab, ts, ls, sd);
      else run_forward(ctx, ab, fa, ls, l);
      if (compute_grads && ctx->multi_stream) BRL_CUDA(cudaStreamWaitEvent(ls, ln.ev_zero, 0));
      if (fused) fused_tail(ctx, ab, ts, fa, y, (float)(c_nll / particles), compute_grads, ab0.acc, ls);
      else launch_nll_elbo(outp, y, B, (float)(c_nll / particles), ab0.acc, compute_grads ? ab.grad[n.out_buf] : nullptr, ls);
      if (compute_grads) {
        BwdArgs ba{x, B, mode, mode == BRL_MODE_WS ? ab.wsamp : mu, sigma, ab.wsamp, 0.f, &nz, sin_.data(), sout_.data(), outp, ab.g0, ab.g1};
        if (fused) fused_backward(ctx, ab, ts, ls, sd);
        else run_backward(ctx, ab, ba, ls, l);
      }
    }
    if (nl > 1) {
      BRL_CUDA(cudaEventRecord(ctx->ev_lane_join, ctx->lane1_main));
      BRL_CUDA(cudaStreamWaitEvent(st, ctx->ev_lane_join, 0));
    }
    for (int l = 0; l < nl; ++l) {
      const int pt = p0 + l;
      const ActBufs& ab = *lanes[l];
      Finalize f{};
      f.P = n.P; f.mode = mode; f.guide = guide; f.first = pt == 0;
      f.mu = mu; f.sigma = sigma; f.w = ab.wsamp; f.delta = ab.delta;
      f.g0 = compute_grads ? ab.g0 : nullptr; f.g1 = compute_grads ? ab.g1 : nullptr;
      f.prior_loc = prior_loc; f.prior_scale = prior_scale; f.c_kl = (float)(cc / particles);
      f.grad_mu = compute_grads ? grad_mu : nullptr; f.grad_sigma = compute_grads ? grad_sigma : nullptr;
      f.grad_log_sigma = (compute_grads && pt == particles - 1) ? grad_log_sigma : nullptr;  // the last particle completes the sum
      f.kl_acc = ab0.acc + 2;
      f.members = (int)M; f.kl_stride = 4;
      launch_finalize(f, st);
    }
  }
  launch_post_scalars(scalars, ab0.acc, c_nll, cc, particles, B, st, (int)M);
  BRL_CUDA(cudaGetLastError());
  return BRL_OK;
}

static bool noise_is_native(const brl_noise* nz) {
  if (!nz) return true;
  if (nz->weight_eps || nz->radial_r) return false;
  for (int l = 0; l < BRL_MAX_LAYERS; ++l)
    if (nz->lrt_eps[l] || nz->flip_in[l] || nz->flip_out[l] || nz->drop_mask[l]) return false;
  return true;
}

int brl_set_step_graph(brl_ctx* ctx, int enable) {
  BRL_REQUIRE(ctx, "brl_set_step_graph: NULL context");
  ctx->graph_enabled = enable != 0;
  return BRL_OK;
}

// brl_elbo_step (M = 1) and brl_elbo_step_ensemble: M members in one chain of launches where fused_ok holds, else one member
// after another on the single-member step
static int elbo_step(brl_ctx* ctx, const float* x, const float* y, int64_t M, int64_t B, const float* mu, const float* sigma,
                     int mode, int guide, int particles, float prior_loc, float prior_scale, int64_t dataset_size,
                     const brl_noise* noise, int compute_grads, double* scalars, float* grad_mu, float* grad_sigma,
                     float* grad_log_sigma, float* out, void* workspace, size_t workspace_bytes, cudaStream_t st,
                     bool graphs = true) {
  const NetSpec& n = *ctx->net;
  Carve c(workspace, workspace_bytes);
  ActBufs ab;
  carve_forward(n, c, B, 1, ab);
  carve_train(n, c, B, ab);
  if (!c.ok) return fail(BRL_ERR_WORKSPACE, std::string(M == 1 ? "brl_elbo_step" : "brl_elbo_step_ensemble") +
                                                ": workspace too small; need " + std::to_string(brl_workspace_bytes(ctx, B, 1, 1, 0)) + " bytes");
  ActBufs ab1;
  int n_lanes = 1;
  if (M > 1) {  // the members' lanes right behind lane 0 (brl_workspace_bytes(B, M, 4)), or one member after another
    carve_tl(n, c, B, ab);
    carve_members(n, c, B, M, true, ab);
    if (!fused_ok(ctx, ab, M, B) || !signs_one_stride(n, noise, particles)) {
      brl_noise base;
      memset(&base, 0, sizeof(base));
      if (noise) base = *noise;
      for (int64_t m = 0; m < M; ++m) {
        const brl_noise nm = noise_at_sample(n, &base, m * particles, B);  // MC-sample index sample0 + m particles, member m's rows
        const int rc = elbo_step(ctx, x + m * B * 540, y + m * B, 1, B, mu + m * n.P, sigma + m * n.P, mode, guide, particles,
                                 prior_loc, prior_scale, dataset_size, &nm, compute_grads, scalars + 4 * m,
                                 compute_grads ? grad_mu + m * n.P : nullptr, compute_grads ? grad_sigma + m * n.P : nullptr,
                                 (compute_grads && grad_log_sigma) ? grad_log_sigma + m * n.P : nullptr,
                                 out + m * particles * B * 2, workspace, workspace_bytes, st, graphs);
        if (rc != BRL_OK) return rc;
      }
      return BRL_OK;
    }
  } else {
    // a second buffer set, if the workspace has room for it (brl_workspace_bytes(B, S >= 2, train = 1)): two particles at a time
    if (particles > 1) {
      carve_forward(n, c, B, 1, ab1);
      carve_train(n, c, B, ab1);
      if (c.ok) n_lanes = 2;
    }
    carve_tl(n, c, B, ab);
    if (n_lanes == 2) {
      carve_tl(n, c, B, ab1);
      if (!ab1.fused) ab.fused = false;  // both particle lanes run the same back-end
    }
  }
  const ActBufs* lanes[2] = {&ab, &ab1};
  brl_ctx::StepKey key;
  memset(&key, 0, sizeof(key));
  key.B = B; key.dataset_size = dataset_size; key.mode = mode; key.guide = guide; key.particles = particles;
  key.compute_grads = compute_grads; key.backend = ctx->gemm_backend; key.has_log_sigma = grad_log_sigma != nullptr;
  key.members = (int)M;
  key.prior_loc = prior_loc; key.prior_scale = prior_scale; key.mu = mu; key.sigma = sigma; key.ws = workspace;
  key.ws_bytes = workspace_bytes;
  CopyJobs o{};  // staging -> the caller's result tensors (the four doubles travel as eight floats)
  o.dst[0] = reinterpret_cast<float*>(scalars); o.src[0] = reinterpret_cast<const float*>(ab.st_scal); o.n[0] = 8 * M;
  o.dst[1] = out; o.src[1] = ab.st_out; o.n[1] = M * particles * B * 2;
  o.njobs = 2;
  if (compute_grads) {
    o.dst[2] = grad_mu; o.src[2] = ab.st_gmu; o.n[2] = M * n.P;
    o.dst[3] = grad_sigma; o.src[3] = ab.st_gsig; o.n[3] = M * n.P;
    o.njobs = 4;
    if (grad_log_sigma) { o.dst[4] = grad_log_sigma; o.src[4] = ab.st_glog; o.n[4] = M * n.P; o.njobs = 5; }
  }
  auto body = [&](const float* bx, const float* by, const brl_noise* bnoise, bool staged, cudaStream_t bst) {
    return elbo_body(ctx, lanes, n_lanes, bx, by, M, B, mu, sigma, mode, guide, particles, prior_loc, prior_scale, dataset_size,
                     bnoise, compute_grads, staged ? ab.st_scal : scalars,
                     staged ? (compute_grads ? ab.st_gmu : nullptr) : grad_mu,
                     staged ? (compute_grads ? ab.st_gsig : nullptr) : grad_sigma,
                     staged ? ((compute_grads && grad_log_sigma) ? ab.st_glog : nullptr) : grad_log_sigma,
                     staged ? ab.st_out : out, bst);
  };
  return run_step(ctx, key, graphs && noise_is_native(noise) && particles <= GRAPH_MAX_PARTICLES, ab, x, y, M * B, noise, o, body, st);
}

int brl_elbo_step(brl_ctx* ctx, const float* x, const float* y, int64_t B, const float* mu, const float* sigma, int mode,
                  int guide, int particles, float prior_loc, float prior_scale, int64_t dataset_size,
                  const brl_noise* noise, int compute_grads, double* scalars, float* grad_mu, float* grad_sigma,
                  float* grad_log_sigma, float* out, void* workspace, size_t workspace_bytes, void* stream) {
  BRL_REQUIRE(ctx && x && y && mu && sigma && scalars && out && workspace, "brl_elbo_step: NULL argument");
  DeviceGuard dg(ctx->device);
  BRL_REQUIRE(B > 0 && particles > 0 && dataset_size > 0 && prior_scale > 0.f, "brl_elbo_step: bad sizes");
  BRL_REQUIRE(guide == BRL_GUIDE_NORMAL || guide == BRL_GUIDE_RADIAL, "Guide unknown. Choose from 'normal', 'radial'.");
  BRL_REQUIRE(mode == BRL_MODE_WS || mode == BRL_MODE_LRT || mode == BRL_MODE_FLIPOUT, "brl_elbo_step: mode must be WS, LRT or FLIPOUT");
  BRL_REQUIRE(!compute_grads || (grad_mu && grad_sigma), "brl_elbo_step: gradient buffers are NULL");
  if (guide == BRL_GUIDE_RADIAL) mode = BRL_MODE_WS;  // bayesian.py:81-83: radial forces nullcontext
  return elbo_step(ctx, x, y, 1, B, mu, sigma, mode, guide, particles, prior_loc, prior_scale, dataset_size, noise, compute_grads,
                   scalars, grad_mu, grad_sigma, grad_log_sigma, out, workspace, workspace_bytes, (cudaStream_t)stream);
}

int brl_elbo_step_ensemble(brl_ctx* ctx, const float* x, const float* y, int64_t M, int64_t B, const float* mu, const float* sigma,
                           int mode, int guide, int particles, float prior_loc, float prior_scale, int64_t dataset_size,
                           const brl_noise* noise, int compute_grads, double* scalars, float* grad_mu, float* grad_sigma,
                           float* grad_log_sigma, float* out, void* workspace, size_t workspace_bytes, void* stream) {
  BRL_REQUIRE(ctx && x && y && mu && sigma && scalars && out && workspace, "brl_elbo_step_ensemble: NULL argument");
  DeviceGuard dg(ctx->device);
  BRL_REQUIRE(M > 0 && M < (1 << 16) && B > 0 && particles > 0 && dataset_size > 0 && prior_scale > 0.f,
              "brl_elbo_step_ensemble: bad M or sizes");
  BRL_REQUIRE(guide == BRL_GUIDE_NORMAL || guide == BRL_GUIDE_RADIAL, "Guide unknown. Choose from 'normal', 'radial'.");
  BRL_REQUIRE(mode == BRL_MODE_WS || mode == BRL_MODE_LRT || mode == BRL_MODE_FLIPOUT,
              "brl_elbo_step_ensemble: mode must be WS, LRT or FLIPOUT");
  BRL_REQUIRE(!compute_grads || (grad_mu && grad_sigma), "brl_elbo_step_ensemble: gradient buffers are NULL");
  if (guide == BRL_GUIDE_RADIAL) mode = BRL_MODE_WS;  // bayesian.py:81-83: radial forces nullcontext
  return elbo_step(ctx, x, y, M, B, mu, sigma, mode, guide, particles, prior_loc, prior_scale, dataset_size, noise, compute_grads,
                   scalars, grad_mu, grad_sigma, grad_log_sigma, out, workspace, workspace_bytes, (cudaStream_t)stream);
}

// the launches of one heteroscedastic-NN step of M members (every pointer final; M > 1 only where fused_ok holds); captured
// as is by the graph path of hnn_step
static int hnn_body(brl_ctx* ctx, const ActBufs& ab, const float* x, const float* y, int64_t M, int64_t B, const float* theta,
                    float p_dropout, const brl_noise* noise, int compute_grads, double* scalars, float* grad_theta, float* out,
                    cudaStream_t st) {
  const NetSpec& n = *ctx->net;
  brl_noise nz = noise_at_sample(n, noise, 0, B);
  FwdArgs fa{x, B, 1, BRL_MODE_DET, theta, nullptr, nullptr, p_dropout, &nz, nullptr, nullptr, out, false};
  if (fused_ok(ctx, ab, M, B)) {
    // level-fused tcgen05 kernels, one contraction with the deterministic weights; dropout masks in the epilogues; member m on
    // blockIdx.z with its own lane, parameters, gradients and MC-sample index sample0 + m
    const brl_ctx::Lane& ln = ctx->lanes[0];
    const TtSide sd{ln.side[0], ln.ev_fork, ln.ev_join[0]};
    const TtStep ts = fused_step(ctx, ab, fa, M, grad_theta, nullptr, 1);
    BRL_CUDA(cudaMemsetAsync(scalars, 0, 2 * M * sizeof(double), st));
    if (compute_grads) BRL_CUDA(cudaMemsetAsync(grad_theta, 0, sizeof(float) * M * n.P, st));
    fused_forward(ctx, ab, ts, st, sd);
    fused_tail(ctx, ab, ts, fa, y, 0.f, compute_grads, scalars, st);
    if (compute_grads) fused_backward(ctx, ab, ts, st, sd);
    BRL_CUDA(cudaGetLastError());
    return BRL_OK;
  }
  run_forward(ctx, ab, fa, st);
  BRL_CUDA(cudaMemsetAsync(scalars, 0, 2 * sizeof(double), st));
  if (compute_grads) {
    int rc = zero_grads(n, ab, B, st);
    if (rc) return rc;
    BRL_CUDA(cudaMemsetAsync(grad_theta, 0, sizeof(float) * n.P, st));
  }
  launch_nll_hnn(out, y, B, scalars, compute_grads ? ab.grad[n.out_buf] : nullptr, st);
  if (compute_grads) {
    BwdArgs ba{x, B, BRL_MODE_DET, theta, nullptr, nullptr, p_dropout, &nz, nullptr, nullptr, out, grad_theta, nullptr};
    run_backward(ctx, ab, ba, st);
  }
  BRL_CUDA(cudaGetLastError());
  return BRL_OK;
}

// brl_hnn_step (M = 1) and brl_hnn_step_ensemble: M members in one chain of launches where fused_ok holds, else one member
// after another on the single-member step
static int hnn_step(brl_ctx* ctx, const float* x, const float* y, int64_t M, int64_t B, const float* theta, float p_dropout,
                    const brl_noise* noise, int compute_grads, double* scalars, float* grad_theta, float* out,
                    void* workspace, size_t workspace_bytes, cudaStream_t st, bool graphs = true) {
  const NetSpec& n = *ctx->net;
  Carve c(workspace, workspace_bytes);
  ActBufs ab;
  carve_forward(n, c, B, 1, ab);
  carve_train(n, c, B, ab);
  if (!c.ok) return fail(BRL_ERR_WORKSPACE, M == 1 ? "brl_hnn_step: workspace too small" : "brl_hnn_step_ensemble: workspace too small");
  carve_tl(n, c, B, ab);
  carve_members(n, c, B, M, false, ab);
  if (M > 1 && !fused_ok(ctx, ab, M, B)) {
    brl_noise base;
    memset(&base, 0, sizeof(base));
    if (noise) base = *noise;
    for (int64_t m = 0; m < M; ++m) {
      const brl_noise nm = noise_at_sample(n, &base, m, B);  // MC-sample index sample0 + m, injected masks of member m
      const int rc = hnn_step(ctx, x + m * B * 540, y + m * B, 1, B, theta + m * n.P, p_dropout, &nm, compute_grads, scalars + 2 * m,
                              compute_grads ? grad_theta + m * n.P : nullptr, out + m * B * 2, workspace, workspace_bytes, st, graphs);
      if (rc != BRL_OK) return rc;
    }
    return BRL_OK;
  }
  // graph replay of native dropout masks or no dropout
  brl_ctx::StepKey key;
  memset(&key, 0, sizeof(key));
  key.B = B; key.mode = -1 /* HNN */; key.particles = 1; key.compute_grads = compute_grads; key.backend = ctx->gemm_backend;
  key.members = (int)M;
  key.prior_loc = p_dropout; key.mu = theta; key.ws = workspace; key.ws_bytes = workspace_bytes;
  CopyJobs o{};
  o.dst[0] = reinterpret_cast<float*>(scalars); o.src[0] = reinterpret_cast<const float*>(ab.st_scal); o.n[0] = 4 * M;
  o.dst[1] = out; o.src[1] = ab.st_out; o.n[1] = M * B * 2;
  o.njobs = 2;
  if (compute_grads) { o.dst[2] = grad_theta; o.src[2] = ab.st_gmu; o.n[2] = M * n.P; o.njobs = 3; }
  auto body = [&](const float* bx, const float* by, const brl_noise* bnoise, bool staged, cudaStream_t bst) {
    return hnn_body(ctx, ab, bx, by, M, B, theta, p_dropout, bnoise, compute_grads, staged ? ab.st_scal : scalars,
                    staged ? (compute_grads ? ab.st_gmu : nullptr) : grad_theta, staged ? ab.st_out : out, bst);
  };
  return run_step(ctx, key, graphs && noise_is_native(noise), ab, x, y, M * B, noise, o, body, st);
}

int brl_hnn_step(brl_ctx* ctx, const float* x, const float* y, int64_t B, const float* theta, float p_dropout,
                 const brl_noise* noise, int compute_grads, double* scalars, float* grad_theta, float* out,
                 void* workspace, size_t workspace_bytes, void* stream) {
  BRL_REQUIRE(ctx && x && y && theta && scalars && out && workspace, "brl_hnn_step: NULL argument");
  DeviceGuard dg(ctx->device);
  BRL_REQUIRE(B > 0 && p_dropout >= 0.f && p_dropout < 1.f, "brl_hnn_step: bad B or p_dropout");
  BRL_REQUIRE(!compute_grads || grad_theta, "brl_hnn_step: grad_theta is NULL");
  return hnn_step(ctx, x, y, 1, B, theta, p_dropout, noise, compute_grads, scalars, grad_theta, out, workspace, workspace_bytes,
                  (cudaStream_t)stream);
}

int brl_hnn_step_ensemble(brl_ctx* ctx, const float* x, const float* y, int64_t M, int64_t B, const float* theta, float p_dropout,
                          const brl_noise* noise, int compute_grads, double* scalars, float* grad_theta, float* out,
                          void* workspace, size_t workspace_bytes, void* stream) {
  BRL_REQUIRE(ctx && x && y && theta && scalars && out && workspace, "brl_hnn_step_ensemble: NULL argument");
  DeviceGuard dg(ctx->device);
  BRL_REQUIRE(M > 0 && M < (1 << 16) && B > 0 && p_dropout >= 0.f && p_dropout < 1.f, "brl_hnn_step_ensemble: bad M, B or p_dropout");
  BRL_REQUIRE(!compute_grads || grad_theta, "brl_hnn_step_ensemble: grad_theta is NULL");
  return hnn_step(ctx, x, y, M, B, theta, p_dropout, noise, compute_grads, scalars, grad_theta, out, workspace, workspace_bytes,
                  (cudaStream_t)stream);
}

}  // extern "C"

// ---- K training steps per call ----------------------------------------------------------------------------------------------
struct TrainArgs {
  const float *X, *Y;
  long long N;
  const int64_t* idx;
  long long K, M, B, step0;
  uint64_t seed;
  long long sample0, window0;
  double *scalars, *metrics;
};

static int train_args_ok(const char* fn, const TrainArgs& a) {
  BRL_REQUIRE(a.X && a.Y && a.idx && a.scalars && a.metrics, std::string(fn) + ": NULL argument");
  BRL_REQUIRE(a.N > 0 && a.K > 0 && a.M > 0 && a.M < (1 << 16) && a.B > 0 && a.step0 >= 0, std::string(fn) + ": bad N, K, M, B or step0");
  BRL_REQUIRE(((uintptr_t)a.X & 15) == 0, std::string(fn) + ": X must be 16-byte aligned");
  return BRL_OK;
}

// Step k of the call is body(noise, stream): gather -> step -> optimizer -> metrics -> row k.  With graphs on and nobody capturing
// `st`, the first step of a configuration runs eagerly, the second is captured (the Philox key read from the descriptor) and every
// later step, in this call or a later one, is one graph launch.  Every TRAIN_TABLE steps setup(su, stream) fills the table of the
// optimizer's per-step scalars for steps step0 + su.k0 + 1 ... (as the single-step optimizer entry point computes them) and makes
// the one launch that writes the descriptor and that table.  Nothing synchronises the host.
// A step that draws `keys` Philox keys takes keys k + 1 ... keys k + keys of the sequence seed + 0x9E3779B97F4A7C15 i; its body gets
// the first (and derives the others: their captured launches read them from where the step's gather writes them).  graphable =
// false keeps every step eager.
template <class Setup, class Body>
static int train_steps(brl_ctx* ctx, const TrainArgs& a, const brl_ctx::StepKey& key, const TrainBufs& t, Setup setup, Body body,
                       cudaStream_t st, bool graphable = true, int keys = 1) {
  brl_ctx::StepGraph* sg = graphable && ctx->graph_enabled && !stream_capturing(st) ? graph_slot(ctx, key) : nullptr;
  const unsigned long long* dyn = reinterpret_cast<const unsigned long long*>(reinterpret_cast<const char*>(t.d) + offsetof(TrainDesc, dyn));
  TrainSetup su;
  su.d = t.d; su.X = a.X; su.Y = a.Y; su.idx = reinterpret_cast<const long long*>(a.idx); su.scalars = a.scalars; su.metrics = a.metrics;
  su.N = a.N; su.seed = a.seed; su.sample0 = (unsigned long long)a.sample0; su.window0 = (unsigned long long)a.window0;
  for (long long k = 0; k < a.K; ++k) {
    if (k % TRAIN_TABLE == 0) {
      su.k0 = k;
      su.n = (int)std::min<long long>(TRAIN_TABLE, a.K - k);
      setup(su, st);
    }
    if (sg && !sg->exec && !sg->bad && sg->seen >= 1)
      capture_step(ctx, sg, dyn, [&](cudaStream_t cs) {
        brl_noise zero;
        memset(&zero, 0, sizeof(zero));
        return body(&zero, cs);
      });
    if (sg && sg->exec) {
      count_launch(sg->launches);
      BRL_CUDA(cudaGraphLaunch(sg->exec, st));
    } else {
      brl_noise nz;
      memset(&nz, 0, sizeof(nz));
      nz.seed = a.seed + 0x9E3779B97F4A7C15ull * (uint64_t)(keys * k + 1);
      nz.sample0 = a.sample0;
      nz.window0 = a.window0;
      const int rc = body(&nz, st);
      if (rc != BRL_OK) return rc;
    }
    if (sg) ++sg->seen;
  }
  BRL_CUDA(cudaGetLastError());
  return BRL_OK;
}

// ClippedAdam's table: the step sizes brl_clipped_adam{,_vi} computes
static auto clipped_adam_setup(float lr, float lrd, float beta1, float beta2, long long step0) {
  return [=](TrainSetup& su, cudaStream_t st) {
    for (int i = 0; i < su.n; ++i) su.steps[i] = adam_step_size(lr, lrd, beta1, beta2, step0 + su.k0 + i + 1);
    launch_train_setup(su, st);
  };
}

// the logged step metrics of M members from their (loc, scale) pairs at src + m mstride, then row k of the results
static void train_metrics_tail(const TrainBufs& t, const float* src, long long mstride, long long M, long long B, int nscal,
                               cudaStream_t st) {
  launch_split_pred(src, mstride, (int)M, B, t.pred, t.std, st);
  launch_test_metrics(t.pred, t.std, t.yb, B, t.met, t.hist, st, 5, (int)M);
  launch_train_tail(t.d, t.scal, nscal, t.met, (int)M, st);
}

// the most hnn_step carves from its workspace for M members of B windows (every optional image included)
static size_t hnn_step_bytes(const NetSpec& n, long long M, long long B) {
  Carve c(nullptr, 0);
  ActBufs ab;
  carve_forward(n, c, B, 1, ab);
  carve_train(n, c, B, ab);
  carve_tl(n, c, B, ab);
  carve_members(n, c, B, M, false, ab);
  return c.used;
}

// brl_hnn_train_steps (kind 6: ClippedAdam) and brl_hnn_train_steps_adam (kind 7: torch's Adam), which differ in the optimizer
// alone.  `opt` holds the float operands the optimizer launch bakes into a captured step; with `kind` they join the graph key, so
// neither call replays the other's graph.  setup(su, col2, stream) writes the descriptor and its table (an Adam call also the second
// column col2), optim(bufs, col2, stream) is step 2 of step k.  Torch's Adam keeps its sqrt(1 - beta2^t) column of TRAIN_TABLE floats
// in front of the step's workspace: brl_workspace_bytes(B, M, 6) leaves the HNN step more than that beyond what it carves (code 3
// adds 4 KB, code 1 at M = 1 a [P] weight sample and the moment state the step does not use).
template <class Setup, class Optim>
static int hnn_train_steps(brl_ctx* ctx, const char* fn, const TrainArgs& a, float* theta, const float* exp_avg, const float* exp_avg_sq,
                           float p_dropout, int kind, const float opt[5], void* workspace, size_t workspace_bytes, Setup setup,
                           Optim optim, cudaStream_t st) {
  if (int rc = train_args_ok(fn, a)) return rc;
  BRL_REQUIRE(p_dropout >= 0.f && p_dropout < 1.f, std::string(fn) + ": bad p_dropout");
  const long long M = a.M, B = a.B;
  const int64_t need = brl_workspace_bytes(ctx, B, M, 6, 0);
  if ((int64_t)workspace_bytes < need)
    return fail(BRL_ERR_WORKSPACE, std::string(fn) + ": workspace too small; need " + std::to_string(need) + " bytes");
  const NetSpec& n = *ctx->net;
  Carve c(workspace, workspace_bytes);
  TrainBufs t;
  carve_train_steps(n, c, M, B, false, t);
  float* col2 = kind == 7 ? c.take<float>(TRAIN_TABLE) : nullptr;
  char* sws = (char*)workspace + c.used;
  const size_t sws_bytes = workspace_bytes - c.used;
  if (col2 && (!c.ok || hnn_step_bytes(n, M, B) > sws_bytes))
    return fail(BRL_ERR_WORKSPACE, std::string(fn) + ": workspace too small for the optimizer's table");
  brl_ctx::StepKey key;
  memset(&key, 0, sizeof(key));
  key.B = B; key.mode = -1 /* HNN */; key.particles = 1; key.compute_grads = 1; key.backend = ctx->gemm_backend;
  key.members = (int)M; key.prior_loc = p_dropout; key.mu = theta; key.ws = workspace; key.ws_bytes = workspace_bytes; key.train = kind;
  memcpy(key.opt, opt, sizeof(key.opt));
  key.state[0] = exp_avg; key.state[1] = exp_avg_sq;
  auto body = [&](const brl_noise* nz, cudaStream_t s) {
    launch_train_gather(t.d, t.xb, t.yb, M * B, s);
    const int rc = hnn_step(ctx, t.xb, t.yb, M, B, theta, p_dropout, nz, 1, t.scal, t.g0, t.out, sws, sws_bytes, s, false);
    if (rc != BRL_OK) return rc;
    optim(t, col2, s);
    train_metrics_tail(t, t.out, B * 2, M, B, 2, s);
    BRL_CUDA(cudaGetLastError());
    return BRL_OK;
  };
  return train_steps(ctx, a, key, t, [&](TrainSetup& su, cudaStream_t s) { setup(su, col2, s); }, body, st);
}

extern "C" {

int brl_elbo_train_steps(brl_ctx* ctx, const float* X, const float* Y, int64_t N, const int64_t* idx, int64_t K, int64_t M, int64_t B,
                         float* loc, float* log_scale, float* scale, float* m_loc, float* v_loc, float* m_log_scale,
                         float* v_log_scale, int64_t step0, float lr, float beta1, float beta2, float eps, float clip_norm, float lrd,
                         float weight_decay, int mode, int guide, int particles, float prior_loc, float prior_scale,
                         int64_t dataset_size, uint64_t seed, int64_t sample0, int64_t window0, double* scalars, double* metrics,
                         void* workspace, size_t workspace_bytes, void* stream) {
  BRL_REQUIRE(ctx && loc && log_scale && scale && m_loc && v_loc && m_log_scale && v_log_scale && workspace,
              "brl_elbo_train_steps: NULL argument");
  DeviceGuard dg(ctx->device);
  const TrainArgs a{X, Y, N, idx, K, M, B, step0, seed, sample0, window0, scalars, metrics};
  if (int rc = train_args_ok("brl_elbo_train_steps", a)) return rc;
  BRL_REQUIRE(particles > 0 && particles <= GRAPH_MAX_PARTICLES && dataset_size > 0 && prior_scale > 0.f,
              "brl_elbo_train_steps: bad particles (1 to 8), dataset size or prior scale");
  BRL_REQUIRE(guide == BRL_GUIDE_NORMAL || guide == BRL_GUIDE_RADIAL, "Guide unknown. Choose from 'normal', 'radial'.");
  BRL_REQUIRE(mode == BRL_MODE_WS || mode == BRL_MODE_LRT || mode == BRL_MODE_FLIPOUT, "brl_elbo_train_steps: mode must be WS, LRT or FLIPOUT");
  if (guide == BRL_GUIDE_RADIAL) mode = BRL_MODE_WS;  // bayesian.py:81-83: radial forces nullcontext
  const int64_t need = brl_workspace_bytes(ctx, B, M, 5, 0);
  if ((int64_t)workspace_bytes < need)
    return fail(BRL_ERR_WORKSPACE, "brl_elbo_train_steps: workspace too small; need " + std::to_string(need) + " bytes");
  const NetSpec& n = *ctx->net;
  Carve c(workspace, workspace_bytes);
  TrainBufs t;
  carve_train_steps(n, c, M, B, true, t);
  char* sws = (char*)workspace + c.used;
  const size_t sws_bytes = workspace_bytes - c.used;
  brl_ctx::StepKey key;
  memset(&key, 0, sizeof(key));
  key.B = B; key.dataset_size = dataset_size; key.mode = mode; key.guide = guide; key.particles = particles;
  key.compute_grads = 1; key.backend = ctx->gemm_backend; key.has_log_sigma = 1; key.members = (int)M;
  key.prior_loc = prior_loc; key.prior_scale = prior_scale; key.mu = loc; key.sigma = scale; key.ws = workspace;
  key.ws_bytes = workspace_bytes; key.train = 5;
  const float opt[5] = {beta1, beta2, eps, clip_norm, weight_decay};
  memcpy(key.opt, opt, sizeof(opt));
  const void* state[5] = {log_scale, m_loc, v_loc, m_log_scale, v_log_scale};
  memcpy(key.state, state, sizeof(state));
  auto body = [&](const brl_noise* nz, cudaStream_t s) {
    launch_train_gather(t.d, t.xb, t.yb, M * B, s);
    const int rc = elbo_step(ctx, t.xb, t.yb, M, B, loc, scale, mode, guide, particles, prior_loc, prior_scale, dataset_size, nz, 1,
                             t.scal, t.g0, t.g1, t.g2, t.out, sws, sws_bytes, s, false);
    if (rc != BRL_OK) return rc;
    launch_clipped_adam_vi(loc, log_scale, scale, t.g0, t.g2, m_loc, v_loc, m_log_scale, v_log_scale, M * n.P, t.d, beta1, beta2,
                           eps, clip_norm, weight_decay, s);
    if (particles == 1) {
      train_metrics_tail(t, t.out, B * 2, M, B, 4, s);
    } else {  // BNN._agg: the precision-weighted aggregate of each member's particles
      for (int64_t m = 0; m < M; ++m) launch_aggregate(t.out + m * particles * B * 2, particles, B, t.agg + m * B * 2, s);
      train_metrics_tail(t, t.agg, B * 2, M, B, 4, s);
    }
    BRL_CUDA(cudaGetLastError());
    return BRL_OK;
  };
  return train_steps(ctx, a, key, t, clipped_adam_setup(lr, lrd, beta1, beta2, step0), body, (cudaStream_t)stream);
}

int brl_hnn_train_steps(brl_ctx* ctx, const float* X, const float* Y, int64_t N, const int64_t* idx, int64_t K, int64_t M, int64_t B,
                        float* theta, float* exp_avg, float* exp_avg_sq, int64_t step0, float lr, float beta1, float beta2, float eps,
                        float clip_norm, float lrd, float weight_decay, float p_dropout, uint64_t seed, int64_t sample0,
                        int64_t window0, double* scalars, double* metrics, void* workspace, size_t workspace_bytes, void* stream) {
  BRL_REQUIRE(ctx && theta && exp_avg && exp_avg_sq && workspace, "brl_hnn_train_steps: NULL argument");
  DeviceGuard dg(ctx->device);
  const TrainArgs a{X, Y, N, idx, K, M, B, step0, seed, sample0, window0, scalars, metrics};
  const float opt[5] = {beta1, beta2, eps, clip_norm, weight_decay};
  const long long MP = M * ctx->net->P;
  return hnn_train_steps(ctx, "brl_hnn_train_steps", a, theta, exp_avg, exp_avg_sq, p_dropout, 6, opt, workspace, workspace_bytes,
                         [su0 = clipped_adam_setup(lr, lrd, beta1, beta2, step0)](TrainSetup& su, float*, cudaStream_t s) { su0(su, s); },
                         [=](const TrainBufs& t, const float*, cudaStream_t s) {
                           launch_clipped_adam(theta, t.g0, exp_avg, exp_avg_sq, MP, t.d, beta1, beta2, eps, clip_norm, weight_decay, s);
                         },
                         (cudaStream_t)stream);
}

int brl_hnn_train_steps_adam(brl_ctx* ctx, const float* X, const float* Y, int64_t N, const int64_t* idx, int64_t K, int64_t M,
                             int64_t B, float* theta, float* exp_avg, float* exp_avg_sq, int64_t step0, double lr, double beta1,
                             double beta2, double eps, double weight_decay, float p_dropout, uint64_t seed, int64_t sample0,
                             int64_t window0, double* scalars, double* metrics, void* workspace, size_t workspace_bytes, void* stream) {
  BRL_REQUIRE(ctx && theta && exp_avg && exp_avg_sq && workspace, "brl_hnn_train_steps_adam: NULL argument");
  DeviceGuard dg(ctx->device);
  BRL_REQUIRE(lr >= 0.0 && beta1 >= 0.0 && beta1 < 1.0 && beta2 >= 0.0 && beta2 < 1.0 && eps >= 0.0,
              "brl_hnn_train_steps_adam: bad lr, betas or eps");
  const TrainArgs a{X, Y, N, idx, K, M, B, step0, seed, sample0, window0, scalars, metrics};
  const AdamArgs aa = torch_adam_args(beta1, beta2, eps, weight_decay);
  const float opt[5] = {aa.w1, aa.b2, aa.w2, aa.eps, aa.wd};
  const long long MP = M * ctx->net->P;
  return hnn_train_steps(ctx, "brl_hnn_train_steps_adam", a, theta, exp_avg, exp_avg_sq, p_dropout, 7, opt, workspace, workspace_bytes,
                         [=](TrainSetup& su, float* bc2, cudaStream_t s) {
                           TrainSetupAdam sa;
                           sa.s = su;
                           sa.bc2 = bc2;
                           for (int i = 0; i < su.n; ++i)
                             torch_adam_step(lr, beta1, beta2, step0 + su.k0 + i + 1, &sa.s.steps[i], &sa.bc2_tab[i]);
                           launch_train_setup(sa, s);
                         },
                         [=](const TrainBufs& t, const float* bc2, cudaStream_t s) {
                           launch_adam(theta, t.g0, exp_avg, exp_avg_sq, MP, t.d, bc2, aa, s);
                         },
                         (cudaStream_t)stream);
}

// Batch k: gather -> brl_elbo_step (weight sampling, no gradients) with key 2k + 1 -> brl_sample_weights, brl_forward and (S > 1)
// brl_aggregate_predictions with key 2k + 2 -> step metrics -> row k.  The ELBO step and the predictive share one region of the
// workspace, one after the other.  A captured batch reads its ELBO key from the descriptor (g_dyn of the capture) and its predictive
// key from key2: the sampler is captured with g_dyn pointing there.
int brl_elbo_val_steps(brl_ctx* ctx, const float* X, const float* Y, int64_t N, const int64_t* idx, int64_t K, int64_t B, const float* loc,
                       const float* scale, int guide, int particles, int64_t S, int engine, float prior_loc, float prior_scale,
                       int64_t dataset_size, uint64_t seed, int64_t sample0, int64_t window0, double* scalars, double* metrics,
                       void* workspace, size_t workspace_bytes, void* stream) {
  BRL_REQUIRE(ctx && loc && scale && workspace, "brl_elbo_val_steps: NULL argument");
  DeviceGuard dg(ctx->device);
  const TrainArgs a{X, Y, N, idx, K, 1, B, 0, seed, sample0, window0, scalars, metrics};
  if (int rc = train_args_ok("brl_elbo_val_steps", a)) return rc;
  BRL_REQUIRE(particles > 0 && particles <= GRAPH_MAX_PARTICLES && dataset_size > 0 && prior_scale > 0.f,
              "brl_elbo_val_steps: bad particles (1 to 8), dataset size or prior scale");
  BRL_REQUIRE(S > 0 && S < (1 << 16) && B * 30 < (1ll << 31) / 512, "brl_elbo_val_steps: bad S or B");
  BRL_REQUIRE(guide == BRL_GUIDE_NORMAL || guide == BRL_GUIDE_RADIAL, "Guide unknown. Choose from 'normal', 'radial'.");
  BRL_REQUIRE(engine == BRL_ENGINE_SIMT_FP32 || engine == BRL_ENGINE_TC_FP16, "brl_elbo_val_steps: unknown engine");
  const int64_t need = brl_workspace_bytes(ctx, B, S, 7, engine);
  if ((int64_t)workspace_bytes < need)
    return fail(BRL_ERR_WORKSPACE, "brl_elbo_val_steps: workspace too small; need " + std::to_string(need) + " bytes");
  Carve c(workspace, workspace_bytes);
  TrainBufs t;
  unsigned long long* key2;
  carve_val_steps(c, B, S, t, key2);
  char* rws = (char*)workspace + c.used;
  const size_t rbytes = workspace_bytes - c.used;
  Carve pc(rws, rbytes);
  ValPredict v;
  carve_val_predict(ctx, pc, B, S, engine, v);
  brl_ctx::StepKey key;
  memset(&key, 0, sizeof(key));
  key.B = B; key.dataset_size = dataset_size; key.mode = BRL_MODE_WS; key.guide = guide; key.particles = particles;
  key.compute_grads = 0; key.backend = ctx->gemm_backend; key.members = 1;
  key.prior_loc = prior_loc; key.prior_scale = prior_scale; key.mu = loc; key.sigma = scale; key.ws = workspace;
  key.ws_bytes = workspace_bytes; key.train = 8; key.S = S; key.engine = engine;
  auto body = [&](const brl_noise* nz, cudaStream_t s) {
    launch_val_gather(t.d, t.xb, t.yb, B, key2, s);
    int rc = elbo_step(ctx, t.xb, t.yb, 1, B, loc, scale, BRL_MODE_WS, guide, particles, prior_loc, prior_scale, dataset_size, nz, 0,
                       t.scal, nullptr, nullptr, nullptr, t.out, rws, rbytes, s, false);
    if (rc != BRL_OK) return rc;
    brl_noise nz2 = *nz;
    nz2.seed += 0x9E3779B97F4A7C15ull;
    const unsigned long long* dyn = g_dyn;
    if (dyn) g_dyn = key2;
    rc = brl_sample_weights(ctx, loc, scale, guide, S, &nz2, v.wsamp, nullptr, v.norms, v.norms_bytes, s);
    if (rc == BRL_OK)
      rc = brl_forward(ctx, t.xb, B, S, BRL_MODE_WS, nullptr, nullptr, v.wsamp, 0.f, &nz2, t.out, engine, v.fws, v.fws_bytes, s);
    g_dyn = dyn;
    if (rc != BRL_OK) return rc;
    if (S > 1) launch_aggregate(t.out, S, B, t.agg, s);  // validation_step uses sample 0 as it is for S = 1
    train_metrics_tail(t, S > 1 ? t.agg : t.out, B * 2, 1, B, 4, s);
    BRL_CUDA(cudaGetLastError());
    return BRL_OK;
  };
  const bool graphable = engine != BRL_ENGINE_TC_FP16 || tc_capturable(ctx->tc);
  return train_steps(ctx, a, key, t, [](TrainSetup& su, cudaStream_t s) { su.n = 0; launch_train_setup(su, s); }, body,
                     (cudaStream_t)stream, graphable, 2);
}

int brl_mixture_moments(const float* mu_m, const float* sigma_m, int64_t M, int64_t nn, float* mu, float* sigma, void* stream) {
  BRL_REQUIRE(mu_m && sigma_m && mu && sigma && M > 0 && nn > 0, "brl_mixture_moments: bad argument");
  launch_mixture(mu_m, sigma_m, M, nn, mu, sigma, (cudaStream_t)stream);
  BRL_CUDA(cudaGetLastError());
  return BRL_OK;
}

int brl_test_metrics(const float* pred, const float* std, const float* y, int64_t nn, double* scalars, void* workspace,
                     size_t workspace_bytes, void* stream) {
  BRL_REQUIRE(pred && std && y && scalars && workspace && nn > 0, "brl_test_metrics: bad argument");
  if (workspace_bytes < 1024) return fail(BRL_ERR_WORKSPACE, "brl_test_metrics: workspace must be >= 1024 bytes");
  launch_test_metrics(pred, std, y, nn, scalars, (unsigned int*)workspace, (cudaStream_t)stream);
  BRL_CUDA(cudaGetLastError());
  return BRL_OK;
}

int brl_step_metrics(const float* pred, const float* std, const float* y, int64_t nn, double* scalars, void* workspace,
                     size_t workspace_bytes, void* stream) {
  BRL_REQUIRE(pred && std && y && scalars && workspace && nn > 0, "brl_step_metrics: bad argument");
  if (workspace_bytes < 1024) return fail(BRL_ERR_WORKSPACE, "brl_step_metrics: workspace must be >= 1024 bytes");
  launch_test_metrics(pred, std, y, nn, scalars, (unsigned int*)workspace, (cudaStream_t)stream, 5);
  BRL_CUDA(cudaGetLastError());
  return BRL_OK;
}

int brl_step_metrics_ensemble(const float* pred, const float* std, const float* y, int64_t M, int64_t nn, double* scalars,
                              void* workspace, size_t workspace_bytes, void* stream) {
  BRL_REQUIRE(pred && std && y && scalars && workspace && M > 0 && M < (1 << 16) && nn > 0, "brl_step_metrics_ensemble: bad argument");
  if (workspace_bytes < (size_t)M * 1024)
    return fail(BRL_ERR_WORKSPACE, "brl_step_metrics_ensemble: workspace must be >= M x 1024 bytes");
  launch_test_metrics(pred, std, y, nn, scalars, (unsigned int*)workspace, (cudaStream_t)stream, 5, (int)M);
  BRL_CUDA(cudaGetLastError());
  return BRL_OK;
}

int brl_clipped_adam(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t nn, int64_t step, float lr,
                     float beta1, float beta2, float eps, float clip_norm, float lrd, float weight_decay, void* stream) {
  BRL_REQUIRE(param && grad && exp_avg && exp_avg_sq && nn > 0 && step >= 1, "brl_clipped_adam: bad argument");
  launch_clipped_adam(param, grad, exp_avg, exp_avg_sq, nn, adam_step_size(lr, lrd, beta1, beta2, step), beta1, beta2, eps,
                      clip_norm, weight_decay, (cudaStream_t)stream);
  BRL_CUDA(cudaGetLastError());
  return BRL_OK;
}

int brl_adam(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t nn, int64_t step, double lr, double beta1,
             double beta2, double eps, double weight_decay, void* stream) {
  BRL_REQUIRE(param && grad && exp_avg && exp_avg_sq && nn > 0 && step >= 1, "brl_adam: bad argument");
  BRL_REQUIRE(lr >= 0.0 && beta1 >= 0.0 && beta1 < 1.0 && beta2 >= 0.0 && beta2 < 1.0 && eps >= 0.0, "brl_adam: bad lr, betas or eps");
  float ss, bc2;
  torch_adam_step(lr, beta1, beta2, step, &ss, &bc2);
  launch_adam(param, grad, exp_avg, exp_avg_sq, nn, ss, bc2, torch_adam_args(beta1, beta2, eps, weight_decay), (cudaStream_t)stream);
  BRL_CUDA(cudaGetLastError());
  return BRL_OK;
}

int brl_clipped_adam_vi_scaled(float* loc, float* log_scale, float* scale, const float* grad_loc, const float* grad_log_scale,
                               float* m_loc, float* v_loc, float* m_log_scale, float* v_log_scale, int64_t nn, int64_t step, float lr,
                               float beta1, float beta2, float eps, float clip_norm, float lrd, float weight_decay, float grad_scale,
                               void* stream) {
  BRL_REQUIRE(loc && log_scale && scale && grad_loc && grad_log_scale && m_loc && v_loc && m_log_scale && v_log_scale && nn > 0 && step >= 1,
              "brl_clipped_adam_vi_scaled: bad argument");
  launch_clipped_adam_vi(loc, log_scale, scale, grad_loc, grad_log_scale, m_loc, v_loc, m_log_scale, v_log_scale, nn,
                         adam_step_size(lr, lrd, beta1, beta2, step), beta1, beta2, eps, clip_norm, weight_decay, (cudaStream_t)stream,
                         grad_scale);
  BRL_CUDA(cudaGetLastError());
  return BRL_OK;
}

int brl_clipped_adam_vi(float* loc, float* log_scale, float* scale, const float* grad_loc, const float* grad_log_scale,
                        float* m_loc, float* v_loc, float* m_log_scale, float* v_log_scale, int64_t nn, int64_t step, float lr,
                        float beta1, float beta2, float eps, float clip_norm, float lrd, float weight_decay, void* stream) {
  BRL_REQUIRE(loc && log_scale && scale && grad_loc && grad_log_scale && m_loc && v_loc && m_log_scale && v_log_scale && nn > 0 && step >= 1,
              "brl_clipped_adam_vi: bad argument");
  launch_clipped_adam_vi(loc, log_scale, scale, grad_loc, grad_log_scale, m_loc, v_loc, m_log_scale, v_log_scale, nn,
                         adam_step_size(lr, lrd, beta1, beta2, step), beta1, beta2, eps, clip_norm, weight_decay, (cudaStream_t)stream);
  BRL_CUDA(cudaGetLastError());
  return BRL_OK;
}

}  // extern "C"
