// Level-fused tcgen05 TRAINING kernels of the Inception conv stack (LRT / Flipout ELBO step) -- interface used by brl_api.cu.
// Reference semantics: tyxe.poutine.local_reparameterization / flipout around nets/inception.py:54-61,125-132 under
// svi.step (bayesian.py:146-147); see brl_tc_train.cu for the design.
#pragma once
#include <cstddef>
#include <cuda_runtime.h>

#include "brl_kernels.cuh"

namespace brl {

constexpr int TT_LAYERS = 10;  // conv layers 0..9 of the Inception table (brl_nets.cpp); layers 10 / 11 (fc, head) stay per-layer

// device buffers of one particle lane (carved from the caller's workspace)
struct TtLane {
  unsigned char* ximg;   // [ntile][X0 X1 X2 XP0 XP1 XP2][132 rows][16 B] fp16
  unsigned char* m1;     // [ntile][16 chunks][132][16 B] fp16: module-1 output, 4 branches x 32 channels (27 real)
  unsigned char* t2;     // [ntile][8 chunks] fp16
  unsigned char* t3;
  unsigned char* g[6];   // bf16 gradient images: [0..2] d/dM1 from b1 / b2a / b3a, [3] d/dMaxPool(M1) from b4, [4] d/dT2, [5] d/dT3
  float* rbuf;           // LRT: eps / (2 sd) of every conv layer output, [layer][ntile][NP][128 rows]
  unsigned char* blob;   // weight images of this step / particle
  float* part;           // weight-gradient partials of the backward CTA groups: [group][layer blocks] (tt_reduce_kernel sums them)
  // fc layer operands, per 128-window M-tile [300 k-chunks][128 windows][16 B], k' = t * 80 + c:
  unsigned char* fimg;   // fp16 module-2 output (features)
  unsigned char* fbimg;  // the same in bf16 (A operand of the weight-gradient GEMM)
  unsigned char* f2img;  // second operand of the forward GEMM: bf16 f^2 (LRT) or fp16 f * s_in (Flipout)
  unsigned char* f2bimg; // Flipout: bf16 f * s_in (A operand of the perturbation-path weight gradient)
  unsigned char* gfimg;  // bf16 gradient w.r.t. the features (written by the fc input-gradient kernel)
  unsigned char* fcblob; // fc weight images [300][64][8]: fp16 mu | bf16 mu | bf16 sigma^2 or (W - mu) | fp16 of the same
};
size_t tt_lane_bytes(long long B);  // a multiple of 256: lanes carved back to back are tt_lane_bytes(B) apart
void tt_carve(unsigned char* base, long long B, TtLane& ln);

struct TtStep {
  const float* x;        // [B,30,18]
  long long B;
  int mode;              // BRL_MODE_LRT / BRL_MODE_FLIPOUT (dual contraction) or BRL_MODE_DET / BRL_MODE_WS (one contraction with the
                         // weights `mu`: the HNN / MC-dropout step, the weight-sampling ELBO of the radial guide)
  const float* mu;       // [P]
  const float* sigma;    // [P]  (LRT)
  const float* wsamp;    // [P]  (Flipout: the particle's weight draw)
  NoiseRef eps[TT_LAYERS];          // LRT eps streams (injected tensor [B, N*30] or Philox)
  const float* sgn_in[TT_LAYERS];   // Flipout [B, Cin]
  const float* sgn_out[TT_LAYERS];  // Flipout [B, Cout]
  NoiseRef drop[TT_LAYERS];         // single-contraction modes: dropout site behind each conv layer (masks [B, N, 30] or Philox)
  float keep[TT_LAYERS];            // its keep probability (1 = no site / dropout off)
  const float* sgn_fc_in;  // Flipout: s_in of the fc layer [B, 2400]
  long long w_off_fc, b_off_fc;
  float* g0;             // flat gradient accumulators [P] (brl_kernels.cuh: Finalize): mean path / variance or perturbation path
  float* g1;
  long long w_off[TT_LAYERS], b_off[TT_LAYERS];
  // Inception: `members` independent nets (the members of a deep ensemble, the seeds of a BNN experiment) in the same launches,
  // member m on blockIdx.z.  Member m reads x + m B 540, mu / sigma / wsamp + m P, its lane images at lane + m lane_stride bytes,
  // and writes g0 / g1 + m P; its noise streams (LRT eps, dropout masks) are the injected tensors + m noise_stride B per_window or
  // Philox with MC-sample index sample0 + m noise_stride, its sign tensors sgn_in / sgn_out / sgn_fc_in + m sign_stride B C.  The
  // tail's y / out / acc / part / dpre / dsec follow (TtTail).
  int members = 1;
  long long P = 0;            // floats between members' parameters / gradients
  long long lane_stride = 0;  // bytes between members' TtLane images (tt_carve of M lanes back to back)
  int noise_stride = 1;       // MC samples between members: 1 (HNN step), `particles` (ELBO step: member-major, particle-minor)
  int sign_stride = 1;        // sign-tensor rows [B, C] between members: 1 (generated per member), `particles` (injected)
};
// forward of the ten conv layers: x -> feature images (+ the activation / eps images the backward pass re-reads); 6 launches
// side stream + two events of the calling lane: independent kernels of a step (weight packing next to the window packing, the fc
// weight gradient next to the conv backward chain) fork to `side` and join back; all of it is stream-capturable
struct TtSide { cudaStream_t side; cudaEvent_t fork, join; };
void tt_forward(const TtLane& ln, const TtStep& s, cudaStream_t st, const TtSide& sd);
// fc layer GEMMs on the tensor pipe.  Forward: both contractions as split-K partial sums into `part` ([2][B][64] fp32, the
// split-K scratch layout of brl_gemm.cu) -- the per-layer engine's split-K epilogue then applies bias / eps * sqrt(var) / signs /
// ReLU.  Backward: dpre / dsec = compact [B, 64] gradients (bwd_act_kernel) -> feature-gradient image + g0 / g1 of the fc layer.
void tt_fc_forward(const TtLane& ln, const TtStep& s, float* part, cudaStream_t st);
void tt_fc_backward(const TtLane& ln, const TtStep& s, const float* dpre, const float* dsec, cudaStream_t st, const TtSide& sd);
// Everything between the fc GEMM and the fc layer's backward GEMMs in ONE launch: fc epilogue over `part`, head forward, softplus /
// threshold, ELBO likelihood (+ its sums in acc[0..1]), head backward (its weight gradients into g0 / g1) and the fc layer's
// activation backward (dpre / dsec, compact [B, 64]).
struct TtTail {
  const float* part;
  const float* y;
  float gscale;           // c_nll / particles (launch_nll_elbo)
  int compute_grads;
  double* acc;
  float* out;             // [B,2]
  float *dpre, *dsec;
  NoiseRef eps_fc, eps_head;
  const float *sout_fc, *sin_head, *sout_head;
  long long hw_off, hb_off;  // flat offsets of the head layer's weight / bias
  int loss_kind = 0;         // single-contraction modes: 0 ELBO likelihood, 1 F.gaussian_nll_loss (HNN step)
  float keep_fc = 1.0f;      // dropout site behind the fc layer
  NoiseRef drop_fc{};
  int width = 64;            // hidden units in front of the head: 64 (Inception fc layer), 32 (Linear layer 3), 320 (Conv-D3: the
                             // pooled conv3 features, given in `part` as [B, 320]; their gradient goes to `dpre`)
  int acc_stride = 2;        // TtStep::members: doubles between members' accumulators (HNN [M][2] = {loss, mse}; ELBO [M][4] =
                             // {nll, squared error, kl, -}); out is [members][noise_stride][B][2], part / dpre / dsec per member
};
void tt_tail(const TtStep& s, const TtTail& t, cudaStream_t st);
// backward: feature-gradient image -> g0 / g1 of the ten conv layers (accumulated: the buffers must be zeroed); 4 launches
void tt_backward(const TtLane& ln, const TtStep& s, cudaStream_t st, const TtSide& sd);
// debug: device buffer int64[6 launches][4 layers][16] receiving clock64 stamps of CTA (0, layer) of the three forward and three
// backward level launches (nullptr = off)
void tt_trace(long long* device_buf);
int tt_status();  // 0 ok; else the code of the first bounded mbarrier wait that timed out (synchronises)

// ---- Linear net (brl_tc_train_linear.cuh): the four hidden layers on the tensor pipe, the head in tt_tail (width 32).
// A TtStep describes the step with the hidden layers at indices 0..3 (eps, sgn_in / sgn_out, drop / keep, w_off / b_off; sgn_in[4]
// = the head's s_in) and w_off_fc / b_off_fc = layer 3, the layer whose epilogue the tail runs.
struct TlLane {
  unsigned char* act[4][4];  // input images of hidden layer l, [M-tile][K/8 chunks][128 windows][16 B]: fp16 a | bf16 a |
                             // bf16 a^2 (LRT) or fp16 a * s_in (Flipout) | bf16 a * s_in (Flipout)
  unsigned char* w[4];       // weight images of hidden layer l, [N/32 slices][K/8][32][16 B]: fp16 mu | bf16 mu |
                             // bf16 sigma^2 or (W - mu) | fp16 (W - mu)
  float* rbuf[3];            // LRT: eps / (2 sd) of hidden layers 0..2 [B, N]
  float* part;               // layer 3's sums for the tail [2][B][32]
};
size_t tl_lane_bytes(long long B);
void tl_carve(unsigned char* base, long long B, TlLane& ln);
// window / weight packing + the four forward launches (layer 3 leaves its sums in ln.part for tt_tail with width 32)
void tl_forward(const TlLane& ln, const TtStep& s, cudaStream_t st, const TtSide& sd);
// dpre / dsec[l]: compact [B, N_l] gradients of hidden layer l ([3] written by tt_tail); writes [0..2] and g0 / g1 of the four
// hidden layers (plain stores)
void tl_backward(const TlLane& ln, const TtStep& s, float* const* dpre, float* const* dsec, cudaStream_t st, const TtSide& sd);

// ---- Conv-D3 net (brl_tc_train_convd3.cuh): the three convs on the tensor pipe as GEMMs over (window, position) rows, the head in
// tt_tail (width 320: features in `feat`, their gradient to `dfeat`).  A TtStep describes the step with the convs at indices 0..2
// (eps, sgn_in / sgn_out, drop / keep, w_off / b_off) and sgn_in[3] = the head's s_in.
struct Tc3Lane {
  unsigned char* img[3][4];  // im2col images of conv l's input, [M-tile][K/8 chunks][128 rows][16 B]: fp16 a | bf16 a |
                             // bf16 a^2 (LRT) or fp16 a * s_in (Flipout) | bf16 a * s_in (Flipout)
  unsigned char* w[3];       // weight images of conv l, [N/32 slices][K/8][32][16 B] (four roles as TlLane::w)
  float* act[3];             // conv l's activation after ReLU / dropout [B * P, N]
  float* rbuf[3];            // LRT: eps / (2 sd) [B * P, N]
  float* g[3][2];            // gradients w.r.t. conv l's pre-activation / second path [B * P, N]
  float* col[2];             // column gradients of conv3 / conv2 (input-gradient GEMMs, mean / second path) [B * 25, 320]
  float* feat;               // pooled conv3 features [B, 320] (tt_tail's `part`)
  float* dfeat;              // their gradient (tt_tail's `dpre`)
};
size_t tc3_lane_bytes(long long B);
void tc3_carve(unsigned char* base, long long B, Tc3Lane& ln);
// weight packing + 3 x (im2col, forward) + the pool into ln.feat
void tc3_forward(const Tc3Lane& ln, const TtStep& s, cudaStream_t st, const TtSide& sd);
// from ln.dfeat (written by tt_tail): g0 / g1 of the three convs (accumulated: the buffers must be zeroed)
void tc3_backward(const Tc3Lane& ln, const TtStep& s, cudaStream_t st, const TtSide& sd);

}  // namespace brl
