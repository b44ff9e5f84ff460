// Level-fused tcgen05 training kernels of the Inception conv stack: the LRT / Flipout forward and backward of the ten conv layers
// that svi.step runs under `fit_ctxt` (bayesian.py:146-147; tyxe local_reparameterization / flipout, SURVEY A.3 / A.4).
//
// Why "level-fused": a 256-window minibatch is 64 tiles of 4 windows (128 rows = 4 x (30 steps + 2 dead rows)).  A CTA owns ONE conv
// layer of ONE tile (forward) or of a few tiles (backward): its operands are whole, MMA-addressable IMAGES
//     activation image of a tile   [8-channel chunk][132 rows][8 x 16 bit]     (2 zero pad rows above / below the 128 tile rows)
//     weight image of a layer      [tap][8-channel chunk][N][8 x 16 bit]
// that travel by cp.async.bulk, so there is no im2col gather anywhere: `padding='same'` is a +-16-byte shift of the A
// descriptor, and the SAME images serve the transposed contractions of the backward pass through MN-major descriptors
// (tools/ubench/umma_probe.cu pins the descriptor semantics on hardware):
//     forward           D[row, n]  = sum_c  act[c, row + tap] * W[n, c, tap]      A K-major (act image),   B K-major (weight image)
//     input gradient    D[row, c]  = sum_n  g[n, row - tap]   * W[n, c, tap]      A K-major (grad image),  B MN-major (weight image^T)
//     weight gradient   D[c, n]    = sum_r  act[c, r + tap]   * g[n, r]           A MN-major (act image^T), B MN-major (grad image^T)
// Every layer is a DUAL contraction into two TMEM accumulators:
//     LRT      mean = a * mu,  var = a^2 * sigma^2,  out = relu(mean + b + eps * sqrt(var + sigma_b^2))        (eps: Philox / injected)
//     Flipout  mean = a * mu,  pert = (a . s_in) * (W - mu),  out = relu(mean + pert . s_out + b_sampled)
// The second operand (a^2 or a . s_in) is built in shared memory from the first by the CTA's threads.  The max-pool in front of the
// two pooled branches is applied by the consumer on its staged input.  Layers of one dependency level run in ONE launch
// (grid = tiles x layers); activations go from level to level as fp16 images through L2, gradients as bf16 images.
// Precision: mean path fp16 x fp16 (10-bit mantissa) in the forward pass, everything else bf16 x bf16 (gradients need fp32's
// exponent range: they carry the 1 / (B * 540) ELBO scale), fp32 accumulation in TMEM.  Stated bound vs the fp32 engine /
// the oracle: outputs 1e-2, loss 5e-3, gradient cosine > 0.999 (tests/test_gpu_tc_train.py).
// The 2400 -> 64 fc layer and the head stay on the per-layer engine (fp32), fed by the fp32 feature buffer written here.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <atomic>
#include <cstdint>

#include "../../include/bayesrul_b200.h"
#include "brl_gemm_epi.cuh"
#include "brl_kernels.cuh"
#include "brl_philox.cuh"
#include "brl_tc_ptx.cuh"
#include "brl_tc_train.cuh"

namespace brl {

extern std::atomic<long long> g_launch_count;

namespace {

constexpr int ROWS = 132, CS = ROWS * 16, ROW0 = 2;
constexpr int TT_PLAIN = 0;  // single contraction: deterministic weights (HNN / MC-dropout) or one weight draw (weight-sampling ELBO)
constexpr int NT = 512;  // threads per CTA: 16 warps = 4 TMEM lane quadrants (rows) x 4 column quarters
enum { IN_X = 0, IN_XP = 1, IN_M1 = 2, IN_M1P = 3, IN_T2 = 4, IN_T3 = 5 };
enum { OUT_M1 = 0, OUT_T2 = 1, OUT_T3 = 2, OUT_FEAT = 3 };

struct TtLayer {
  int layer, in, KC, N, NP, T, out, out_c0;  // out_c0: first chunk of an image output / first channel of a feature output
  int cin;                                   // real input channels (torch weight [N, cin, T])
  int w0h, w0b, w1b, w1h, bias, tap_bytes;   // byte offsets inside the weight blob; bytes of one tap's [KC][NP][8] tile
  int gdst;                                  // gradient image receiving this layer's input gradient (-1: input is x)
  int roff_per_tile;                         // float offset of this layer's rbuf block inside a tile's 336 * 128 floats
  int poff;                                  // float offset of this layer's weight-gradient partials inside a group's block:
                                             // [2 paths][N][T][KC * 8 image channels] then [2][64] bias sums
  long long w_off, b_off;                    // flat parameter offsets
};

// static description of the ten conv layers (brl_nets.cpp build_inception order)
struct Table {
  TtLayer L[TT_LAYERS];
  int blob_bytes, pack_start[TT_LAYERS + 1];
  int part_floats;  // floats of one group's partial block (all layers)
};
const Table& table() {
  static const Table t = [] {
    Table tb{};
    const int in_[10] = {IN_X, IN_X, IN_X, IN_XP, IN_M1, IN_M1, IN_T2, IN_M1, IN_T3, IN_M1P};
    const int KC[10] = {4, 4, 4, 4, 16, 16, 8, 16, 8, 16};
    const int N[10] = {27, 27, 27, 27, 16, 64, 16, 64, 16, 32};
    const int T[10] = {1, 3, 5, 3, 1, 1, 3, 1, 5, 1};
    const int out[10] = {OUT_M1, OUT_M1, OUT_M1, OUT_M1, OUT_FEAT, OUT_T2, OUT_FEAT, OUT_T3, OUT_FEAT, OUT_FEAT};
    const int oc0[10] = {0, 4, 8, 12, 0, 0, 16, 0, 32, 48};
    const int cin[10] = {18, 18, 18, 18, 108, 108, 64, 108, 64, 108};
    const int gdst[10] = {-1, -1, -1, -1, 0, 1, 4, 2, 5, 3};
    int off = 0, roff = 0, ps = 0, po = 0;
    for (int i = 0; i < 10; ++i) {
      TtLayer& l = tb.L[i];
      l.layer = i; l.in = in_[i]; l.KC = KC[i]; l.N = N[i]; l.NP = (N[i] + 15) & ~15; l.T = T[i]; l.out = out[i]; l.out_c0 = oc0[i];
      l.cin = cin[i]; l.gdst = gdst[i];
      l.tap_bytes = l.KC * l.NP * 16;
      const int img = l.T * l.tap_bytes;
      l.w0h = off; off += img;
      l.w0b = off; off += img;
      l.w1b = off; off += img;
      l.w1h = off; off += img;
      l.bias = off; off += 2 * 64 * 4;
      l.roff_per_tile = roff; roff += l.NP * 128;
      l.poff = po; po += 2 * l.N * l.T * l.KC * 8 + 128;
      tb.pack_start[i] = ps; ps += l.T * l.KC * 8 * l.NP;
    }
    tb.pack_start[10] = ps;
    tb.blob_bytes = off;
    tb.part_floats = po;
    return tb;
  }();
  return t;
}
constexpr int RBUF_PER_TILE = 336 * 128;  // sum of NP over the ten layers x 128 rows
// fc layer (2400 -> 64): feature images of a 128-window M-tile, [300 k-chunks][128 windows][8 x 16 bit], k' = t * 80 + c
// (chunk = t * 10 + c / 8); weight images [300 k-chunks][64 n][8]
constexpr int FC_KC = 300, FC_CHUNK = 128 * 16, FC_MT_BYTES = FC_KC * FC_CHUNK, FC_WIMG = FC_KC * 64 * 16;
constexpr int FC_KS = 30, FC_KCS = FC_KC / FC_KS;  // forward: K split over 30 CTAs of 10 chunks (5 MMA k-steps) per M-tile
constexpr int FC_NS = 25, FC_NCS = FC_KC / FC_NS;  // input gradient: N' = 2400 in 25 slices of 96 columns (12 chunks) per M-tile
__device__ __forceinline__ long long feat_addr(int gw, int t, int c0) {  // 16-byte unit of window gw, step t, channels [c0, c0 + 8)
  return ((long long)(gw >> 7) * FC_KC + t * 10 + (c0 >> 3)) * FC_CHUNK + (gw & 127) * 16;
}

// image channel k of an input -> real channel of the torch weight / sign tensor (-1: padding channel)
__device__ __forceinline__ int real_ch(int in, int k) {
  if (in <= IN_XP) return k < 18 ? k : -1;
  if (in <= IN_M1P) { const int br = k >> 5, j = k & 31; return j < 27 ? br * 27 + j : -1; }
  return k < 64 ? k : -1;
}
struct RowInfo { int t, gw; bool live; };
__device__ __forceinline__ RowInfo row_info(int rr, int tile, int B) {
  const int r = rr - ROW0;
  RowInfo o;
  o.t = r & 31;
  o.gw = tile * 4 + (r >> 5);
  o.live = r >= 0 && r < 128 && o.t < 30 && o.gw < B;
  return o;
}
__device__ __forceinline__ void unpack_h8(const uint4& v, float (&f)[8]) {
  const __half2* h = reinterpret_cast<const __half2*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float2 t = __half22float2(h[i]); f[2 * i] = t.x; f[2 * i + 1] = t.y; }
}
__device__ __forceinline__ void unpack_b8(const uint4& v, float (&f)[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float2 t = __bfloat1622float2(h[i]); f[2 * i] = t.x; f[2 * i + 1] = t.y; }
}
__device__ __forceinline__ uint4 pack_b8(const float (&f)[8]) {
  uint4 r;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
  return r;
}
__device__ __forceinline__ uint4 pack_h8(const float (&f)[8]) {
  return make_uint4(pack_h2(f[0], f[1]), pack_h2(f[2], f[3]), pack_h2(f[4], f[5]), pack_h2(f[6], f[7]));
}
// kind::f16 instruction descriptor: fp32 D, operand formats (0 fp16, 1 bf16 -- both operands the same: a mixed pair is an
// illegal instruction on B200), majors (1 = MN-major), M = 128
__host__ __device__ constexpr uint32_t tt_idesc(int n, int fmt, int a_mn, int b_mn) {
  return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
         ((uint32_t)(n >> 3) << 17) | ((128u >> 4) << 24);
}
// four normals of one Philox block (brl_philox.cuh::normal4 with hardware log / sin / cos)
__device__ __forceinline__ float4 normal4_fast(const uint4& r) {
  const float rad0 = sqrtf(-2.0f * __logf(u01(r.x))), rad1 = sqrtf(-2.0f * __logf(u01(r.z)));
  float s0, c0, s1, c1;
  __sincosf(6.283185307179586f * u01(r.y), &s0, &c0);
  __sincosf(6.283185307179586f * u01(r.w), &s1, &c1);
  return make_float4(rad0 * c0, rad0 * s0, rad1 * c1, rad1 * s1);
}
// column sums of eight values per lane over the 32 lanes of a warp with 9 shuffles instead of 40: the first three butterfly steps
// exchange HALF of the values each (a lane keeps the half its lane bit selects and adds its partner's), the last two add.  Every
// lane ends up with the total of channel (lane >> 2) & 7.
__device__ __forceinline__ float warp_sum8(const float (&v)[8], int lane) {
  float a[4], b[2], c;
  const bool h4 = lane & 16, h3 = lane & 8, h2 = lane & 4;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float keep = h4 ? v[4 + i] : v[i], send = h4 ? v[i] : v[4 + i];
    a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const float keep = h3 ? a[2 + i] : a[i], send = h3 ? a[i] : a[2 + i];
    b[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
  {
    const float keep = h2 ? b[1] : b[0], send = h2 ? b[0] : b[1];
    c = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  c += __shfl_xor_sync(0xffffffffu, c, 2);
  c += __shfl_xor_sync(0xffffffffu, c, 1);
  return c;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// ensemble member blockIdx.z (TtStep::members): its lane images sit `stride` bytes after the previous member's
__device__ __forceinline__ TtLane member_lane(TtLane ln, long long stride) {
  const long long o = stride * blockIdx.z;
  auto sh = [o](auto* p) { return p ? reinterpret_cast<decltype(p)>(reinterpret_cast<unsigned char*>(p) + o) : p; };
  ln.ximg = sh(ln.ximg); ln.m1 = sh(ln.m1); ln.t2 = sh(ln.t2); ln.t3 = sh(ln.t3);
  for (int k = 0; k < 6; ++k) ln.g[k] = sh(ln.g[k]);
  ln.rbuf = sh(ln.rbuf); ln.blob = sh(ln.blob); ln.part = sh(ln.part);
  ln.fimg = sh(ln.fimg); ln.fbimg = sh(ln.fbimg); ln.f2img = sh(ln.f2img); ln.f2bimg = sh(ln.f2bimg); ln.gfimg = sh(ln.gfimg);
  ln.fcblob = sh(ln.fcblob);
  return ln;
}
// the member's noise stream: `stride` MC samples per member (1 for the HNN step, `particles` for the ELBO step), i.e. injected
// tensors [members * stride, B, per_window] and Philox keys with MC-sample index sample0 + member * stride
__device__ __forceinline__ NoiseRef member_noise(NoiseRef nz, long long per_window, int B, int stride) {
  if (nz.ptr) nz.ptr += (long long)blockIdx.z * stride * B * per_window;
  else nz.sample0 += blockIdx.z * (unsigned)stride;
  return nz;
}
template <typename T>
__device__ __forceinline__ T* member_ptr(T* p, long long stride) { return p ? p + stride * blockIdx.z : p; }

// ------------------------------------------------------------------------------------------------
// window images: fp32 windows -> fp16 chunk images X and XP = MaxPool1d(3,1,1)(X) (-inf padding), pad rows zero
// ------------------------------------------------------------------------------------------------
__global__ void tt_packx_kernel(const float* __restrict__ x, unsigned char* __restrict__ ximg, int B, int ntile, long long lane_stride) {
  const long long u = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (u >= (long long)ntile * 3 * ROWS) return;
  x += (long long)blockIdx.z * B * 540;
  ximg += lane_stride * blockIdx.z;
  const int tile = (int)(u / (3 * ROWS)), v = (int)(u % (3 * ROWS)), c = v / ROWS, rr = v % ROWS;
  const RowInfo ri = row_info(rr, tile, B);
  float f[8], pm[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) f[j] = pm[j] = 0.f;
  if (ri.live) {
    const float* px = x + (long long)ri.gw * 540 + ri.t * 18 + c * 8;
    const int nf = c < 2 ? 8 : 2;
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (j < nf) {
        const float v0 = __half2float(__float2half_rn(px[j]));
        float m = v0;
        if (ri.t > 0) m = fmaxf(m, __half2float(__float2half_rn(px[j - 18])));
        if (ri.t < 29) m = fmaxf(m, __half2float(__float2half_rn(px[j + 18])));
        f[j] = v0;
        pm[j] = m;
      }
  }
  unsigned char* dst = ximg + ((long long)tile * 6 + c) * CS + rr * 16;
  *reinterpret_cast<uint4*>(dst) = pack_h8(f);
  *reinterpret_cast<uint4*>(dst + 3 * CS) = pack_h8(pm);
}

// ------------------------------------------------------------------------------------------------
// weight images of one step / particle
// ------------------------------------------------------------------------------------------------
struct TtPackArgs {
  TtLayer L[TT_LAYERS];
  int start[TT_LAYERS + 1];
  int mode;
  const float *mu, *second;  // second: sigma (LRT) or the weight draw (Flipout)
  unsigned char* blob;
  long long P, lane_stride;  // ensemble members (blockIdx.z): parameter / lane strides
};
__global__ void tt_pack_kernel(const TtPackArgs a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const float* mu = a.mu + a.P * blockIdx.z;
  const float* second = a.second + a.P * blockIdx.z;
  unsigned char* blob = a.blob + a.lane_stride * blockIdx.z;
  if (i < a.start[TT_LAYERS]) {
    int li = 0;
    while (i >= a.start[li + 1]) ++li;
    const TtLayer& l = a.L[li];
    int j = i - a.start[li];
    const int n = j % l.NP; j /= l.NP;
    const int k = j % (l.KC * 8);
    const int tap = j / (l.KC * 8);
    const int cr = real_ch(l.in, k);
    float m = 0.f, s = 0.f;
    if (n < l.N && cr >= 0) {
      const long long wi = l.w_off + ((long long)n * l.cin + cr) * l.T + tap;
      m = mu[wi];
      const float v = second[wi];
      s = a.mode == BRL_MODE_LRT ? v * v : a.mode == BRL_MODE_FLIPOUT ? v - m : 0.f;
    }
    const int o = tap * l.tap_bytes + (k >> 3) * (l.NP * 16) + n * 16 + (k & 7) * 2;
    *reinterpret_cast<__half*>(blob + l.w0h + o) = __float2half_rn(m);
    *reinterpret_cast<__nv_bfloat16*>(blob + l.w0b + o) = __float2bfloat16_rn(m);
    *reinterpret_cast<__nv_bfloat16*>(blob + l.w1b + o) = __float2bfloat16_rn(s);
    *reinterpret_cast<__half*>(blob + l.w1h + o) = __float2half_rn(s);
    return;
  }
  const int b = i - a.start[TT_LAYERS];
  if (b < TT_LAYERS * 64) {
    const TtLayer& l = a.L[b >> 6];
    const int n = b & 63;
    float b0 = 0.f, b1 = 0.f;
    if (n < l.N) {
      if (a.mode == BRL_MODE_LRT) { b0 = mu[l.b_off + n]; const float sb = second[l.b_off + n]; b1 = sb * sb; }
      else if (a.mode == BRL_MODE_FLIPOUT) b0 = second[l.b_off + n];  // Flipout adds the SAMPLED bias (SURVEY A.4)
      else b0 = mu[l.b_off + n];
    }
    float* bias = reinterpret_cast<float*>(blob + l.bias);
    bias[n] = b0;
    bias[64 + n] = b1;
  }
}

// ------------------------------------------------------------------------------------------------
// forward: one CTA = one conv layer of one tile
// ------------------------------------------------------------------------------------------------
constexpr int F_A = 0, F_A2 = 16 * CS, F_W0 = 32 * CS, F_W1 = F_W0 + 16384, F_BIAS = F_W1 + 16384, F_BAR = F_BIAS + 512;
constexpr int F_SMEM = F_BAR + 64;

struct TtFwdArgs {
  TtLane ln;
  int B, ntile, nl;
  TtLayer lay[4];
  NoiseRef eps[4];
  const float* sgn_in[4];
  const float* sgn_out[4];
  const float* sgn_fc_in;  // Flipout: s_in of the fc layer [B, 2400] (the feature producers build its perturbation operand)
  NoiseRef drop[4];        // PLAIN mode: dropout site behind the layer (injected masks [B, N, 30] or Philox)
  float keep[4];           // its keep probability (1 = no dropout site / dropout off)
  long long lane_stride;   // ensemble members (blockIdx.z): bytes between their lanes
  int noise_stride, sign_stride;  // ensemble members: MC samples / sign-tensor rows [B, C] between their noise (TtStep)
  int* status;
  long long* trace;  // debug: clock64 stamps of CTA (0, y), [4 layers][16] (nullptr = off)
};

__device__ __forceinline__ const unsigned char* input_image(const TtLane& ln, int in, int tile) {
  switch (in) {
    case IN_X: return ln.ximg + (long long)tile * 6 * CS;
    case IN_XP: return ln.ximg + (long long)tile * 6 * CS + 3 * CS;
    case IN_M1: case IN_M1P: return ln.m1 + (long long)tile * 16 * CS;
    case IN_T2: return ln.t2 + (long long)tile * 8 * CS;
    default: return ln.t3 + (long long)tile * 8 * CS;
  }
}
__device__ __forceinline__ void bulk_copy_chunked(uint32_t dst, const unsigned char* src, int bytes, uint32_t bar) {
  for (int o = 0; o < bytes; o += 16384) bulk_g2s(dst + o, src + o, min(16384, bytes - o), bar);
}
// MaxPool1d(3,1,1) of a post-ReLU activation image (values >= 0, dead / pad rows are zero, so they act as the -inf padding)
__device__ __forceinline__ void pool_image(const unsigned char* raw, unsigned char* dst, int KC, int tile, int B, int tid) {
  for (int idx = tid; idx < KC * ROWS; idx += NT) {
    const int ch = idx / ROWS, rr = idx - ch * ROWS;
    uint4 o = make_uint4(0, 0, 0, 0);
    if (row_info(rr, tile, B).live) {
      const unsigned char* p = raw + ch * CS + rr * 16;
      o = hmax4(*reinterpret_cast<const uint4*>(p), hmax4(*reinterpret_cast<const uint4*>(p - 16), *reinterpret_cast<const uint4*>(p + 16)));
    }
    *reinterpret_cast<uint4*>(dst + ch * CS + rr * 16) = o;
  }
}
// second operand of the dual contraction from the fp16 activation image: bf16(a^2) (LRT) or a * s_in (Flipout; H16: as fp16 --
// exact -- for the forward pass, whose perturbation GEMM runs fp16 x fp16; bf16 for the backward contractions)
template <int MODE, bool H16>
__device__ __forceinline__ void second_operand(const unsigned char* A, unsigned char* A2, unsigned char* Ab, const TtLayer& L,
                                               const float* sgn_in, int tile, int B, int tid) {
  for (int idx = tid; idx < L.KC * ROWS; idx += NT) {
    const int ch = idx / ROWS, rr = idx - ch * ROWS;
    float f[8], s[8];
    unpack_h8(*reinterpret_cast<const uint4*>(A + ch * CS + rr * 16), f);
    if (Ab) *reinterpret_cast<uint4*>(Ab + ch * CS + rr * 16) = pack_b8(f);
    if (MODE == TT_PLAIN) continue;  // single contraction: only the bf16 copy is needed (backward pass)
    if (MODE == BRL_MODE_LRT) {
#pragma unroll
      for (int j = 0; j < 8; ++j) s[j] = f[j] * f[j];
    } else {
      const RowInfo ri = row_info(rr, tile, B);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int cr = real_ch(L.in, ch * 8 + j);
        s[j] = (ri.live && cr >= 0) ? f[j] * __ldg(sgn_in + (long long)ri.gw * L.cin + cr) : 0.f;
      }
    }
    *reinterpret_cast<uint4*>(A2 + ch * CS + rr * 16) = H16 ? pack_h8(s) : pack_b8(s);
  }
}

template <int MODE>
__global__ void __launch_bounds__(NT, 1) tt_fwd_kernel(const TtFwdArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  const TtLayer& L = a.lay[blockIdx.y];
  const int tile = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  long long* tr = (a.trace && blockIdx.x == 0 && blockIdx.z == 0 && tid == 0) ? a.trace + blockIdx.y * 16 : nullptr;
  const TtLane ln = member_lane(a.ln, a.lane_stride);
  if (tr) tr[0] = clock64();
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar_ld = sbase + F_BAR, bar_mma = bar_ld + 8;
  uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + F_BAR + 16);
  if (tid == 0) {
    mbar_init(bar_ld, 1);
    mbar_init(bar_mma, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc(smem_u32(tslot), 128);
  if (L.in <= IN_XP)  // K = 32 for the 18 input features: the 4th chunk is zero
    for (int i = tid; i < CS / 16; i += NT) reinterpret_cast<uint4*>(smem + F_A + 3 * CS)[i] = make_uint4(0, 0, 0, 0);
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tslot;
  const int ncopy = L.in <= IN_XP ? 3 : L.KC;
  const int img_bytes = L.T * L.tap_bytes;
  if (tid == 0) {
    mbar_expect_tx(bar_ld, ncopy * CS + (MODE == TT_PLAIN ? 1 : 2) * img_bytes + 512);
    bulk_copy_chunked(sbase + (L.in == IN_M1P ? F_A2 : F_A), input_image(ln, L.in, tile), ncopy * CS, bar_ld);
    bulk_copy_chunked(sbase + F_W0, ln.blob + L.w0h, img_bytes, bar_ld);
    if (MODE != TT_PLAIN) bulk_copy_chunked(sbase + F_W1, ln.blob + (MODE == BRL_MODE_FLIPOUT ? L.w1h : L.w1b), img_bytes, bar_ld);
    bulk_g2s(sbase + F_BIAS, ln.blob + L.bias, 512, bar_ld);
  }
  if (tr) tr[1] = clock64();
  mbar_wait(bar_ld, 0, a.status, 40);
  if (tr) tr[2] = clock64();
  if (L.in == IN_M1P) {  // the pooled branch: pool the staged raw image first
    pool_image(smem + F_A2, smem + F_A, L.KC, tile, a.B, tid);
    __syncthreads();
  }
  constexpr bool P1H = MODE == BRL_MODE_FLIPOUT;  // perturbation path: fp16 operands (W - mu is far above fp16's subnormals for q_scale >= 1e-4)
  if (MODE != TT_PLAIN)
    second_operand<MODE, P1H>(smem + F_A, smem + F_A2, nullptr, L,
                              member_ptr(a.sgn_in[blockIdx.y], (long long)a.sign_stride * a.B * L.cin), tile, a.B, tid);
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  if (tr) tr[3] = clock64();
  if (warp == 0) {
    tc_fence_after();
    if (elect_one()) {
      const int pad = (L.T - 1) >> 1;
      for (int tap = 0; tap < L.T; ++tap)
        for (int ks = 0; ks < L.KC / 2; ++ks) {
          const uint32_t ao = 2 * ks * CS + (ROW0 + tap - pad) * 16, wo = tap * L.tap_bytes + 2 * ks * L.NP * 16;
          umma(tmem, umma_desc(sbase + F_A + ao, CS, 128), umma_desc(sbase + F_W0 + wo, L.NP * 16, 128), tt_idesc(L.NP, 0, 0, 0),
               (tap | ks) != 0);
          if (MODE != TT_PLAIN)
            umma(tmem + L.NP, umma_desc(sbase + F_A2 + ao, CS, 128), umma_desc(sbase + F_W1 + wo, L.NP * 16, 128),
                 tt_idesc(L.NP, P1H ? 0 : 1, 0, 0), (tap | ks) != 0);
        }
      umma_commit(bar_mma);
    }
    __syncwarp();
  }
  mbar_wait(bar_mma, 0, a.status, 41);
  tc_fence_after();
  if (tr) tr[4] = clock64();
  // ---- epilogue: thread = tile row (TMEM lane quadrant = warp % 4) x column quarter (warp / 4), eight columns at a time
  const int row = (warp & 3) * 32 + lane, cq = warp >> 2;
  const RowInfo ri = row_info(ROW0 + row, tile, a.B);
  const uint32_t la = tmem + ((uint32_t)((warp & 3) * 32) << 16);
  const float* bias = reinterpret_cast<const float*>(smem + F_BIAS);
  const NoiseRef nz = MODE == BRL_MODE_LRT ? member_noise(a.eps[blockIdx.y], (long long)L.N * 30, a.B, a.noise_stride) : a.eps[blockIdx.y];
  const NoiseKey nk = noise_key(nz);
  const float* sout = member_ptr(a.sgn_out[blockIdx.y], (long long)a.sign_stride * a.B * L.N);
  const NoiseRef dz = MODE == TT_PLAIN ? member_noise(a.drop[blockIdx.y], (long long)L.N * 30, a.B, a.noise_stride) : a.drop[blockIdx.y];
  float* rb = ln.rbuf ? ln.rbuf + (long long)tile * RBUF_PER_TILE + L.roff_per_tile : nullptr;
  unsigned char* oimg = L.out == OUT_M1 ? ln.m1 + (long long)tile * 16 * CS
                        : L.out == OUT_T2 ? ln.t2 + (long long)tile * 8 * CS
                        : L.out == OUT_T3 ? ln.t3 + (long long)tile * 8 * CS : nullptr;
  // LRT eps of the warp's window (one warp = the 30 steps of one window x 8 channels = elements [240 g, 240 g + 240) of the
  // layer's stream, i.e. exactly Philox blocks [60 g, 60 g + 60)): every lane draws two blocks = eight normals into a per-warp
  // scratch (the operand regions are dead once the MMAs have completed) instead of one block per element
  float* scratch = reinterpret_cast<float*>(smem + F_A) + warp * 256;
  for (int g = cq; g < L.NP / 8; g += 4) {
    float v0[8], v1[8], o[8];
    tmem_ld8(la + g * 8, v0);
    if (MODE != TT_PLAIN) tmem_ld8(la + L.NP + g * 8, v1);
    KeepBits kb = {};
    const float keep = MODE == TT_PLAIN ? a.keep[blockIdx.y] : 1.0f;
    const uint32_t e0 = (uint32_t)ri.t * (uint32_t)((L.N + 15) & ~15) + (uint32_t)(g * 8);  // dropout element order: position-major
    if (MODE == TT_PLAIN && keep < 1.0f && !dz.ptr) {  // 8 of the 16 keep decisions of one Philox block
      const NoiseKey dk = noise_key(dz);
      kb = keep_bits(philox_block_mask(dk.seed, dz.kind, dz.site, dk.sample0, dk.window0 + ri.gw, e0 >> 4), keep_threshold(keep));
    }
    if (MODE == BRL_MODE_LRT && !nz.ptr) {
      __syncwarp();
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const int bi = k * 32 + lane;
        if (bi < 60)
          *reinterpret_cast<float4*>(scratch + bi * 4) =
              normal4_fast(philox_block(nk.seed, nz.kind, nz.site, nk.sample0, nk.window0 + ri.gw, (uint32_t)(60 * g + bi)));
      }
      __syncwarp();
    }
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int n = g * 8 + j;
      const bool on = ri.live && n < L.N;
      float pre;
      if (MODE == BRL_MODE_LRT) {
        float var = v1[j] + bias[64 + n];
        if (var < 0.f) var += fabsf(var) + 1e-6f;
        const float sd = sqrtf(var);
        const float e = !on ? 0.f : nz.ptr ? nz.ptr[(long long)ri.gw * (L.N * 30) + n * 30 + ri.t] : scratch[j * 30 + ri.t];
        pre = fmaf(sd, e, v0[j] + bias[n]);
        if (rb) rb[(long long)n * 128 + row] = (on && sd > 0.f) ? e / (2.0f * sd) : 0.f;
      } else if (MODE == BRL_MODE_FLIPOUT) {
        pre = v0[j] + bias[n] + (on ? v1[j] * __ldg(sout + (long long)ri.gw * L.N + n) : 0.f);
      } else {
        pre = v0[j] + bias[n];
      }
      o[j] = on ? fmaxf(pre, 0.f) : 0.f;
      if (MODE == TT_PLAIN && keep < 1.0f && on) {  // dropout site behind the ReLU (inception.py:48-52,119-123)
        const bool kp = dz.ptr ? dz.ptr[((long long)ri.gw * L.N + n) * 30 + ri.t] != 0.f : keep_at(kb, (e0 & 15u) + j);
        o[j] = kp ? o[j] / keep : 0.f;
      }
    }
    if (oimg) {
      *reinterpret_cast<uint4*>(oimg + (L.out_c0 + g) * CS + (ROW0 + row) * 16) = pack_h8(o);
    } else if (ri.live) {  // module-2 output = the fc layer's operands: fp16 features, their bf16 copy and the second operand
      const int c0 = L.out_c0 + g * 8;
      const long long fa = feat_addr(ri.gw, ri.t, c0);
      const uint4 fh = pack_h8(o);
      float fr[8], f2[8];
      unpack_h8(fh, fr);
#pragma unroll
      for (int j = 0; j < 8; ++j)
        f2[j] = MODE == BRL_MODE_LRT ? fr[j] * fr[j]
                : MODE == BRL_MODE_FLIPOUT ? fr[j] * __ldg(a.sgn_fc_in + ((long long)blockIdx.z * a.sign_stride * a.B + ri.gw) * 2400 + (c0 + j) * 30 + ri.t) : 0.f;
      *reinterpret_cast<uint4*>(ln.fimg + fa) = fh;
      *reinterpret_cast<uint4*>(ln.fbimg + fa) = pack_b8(fr);
      if (MODE == BRL_MODE_LRT) {
        *reinterpret_cast<uint4*>(ln.f2img + fa) = pack_b8(f2);
      } else if (MODE == BRL_MODE_FLIPOUT) {  // the perturbation GEMM runs fp16 x fp16 in the forward pass (f * s_in is exact in fp16), bf16 in the backward pass
        *reinterpret_cast<uint4*>(ln.f2img + fa) = pack_h8(f2);
        *reinterpret_cast<uint4*>(ln.f2bimg + fa) = pack_b8(f2);
      }
    }
  }
  if (oimg && tid < 4) {  // the image's pad rows
    const int pr = tid < 2 ? tid : 128 + tid;
    for (int c = 0; c < L.NP / 8; ++c) *reinterpret_cast<uint4*>(oimg + (L.out_c0 + c) * CS + pr * 16) = make_uint4(0, 0, 0, 0);
  }
  tc_fence_before();
  __syncthreads();
  if (tr) tr[5] = clock64();
  if (warp == 0) tmem_dealloc(tmem, 128);
}

// ------------------------------------------------------------------------------------------------
// backward: one CTA = one conv layer of a group of tiles (weight gradients accumulate in TMEM over the group)
// ------------------------------------------------------------------------------------------------
constexpr int B_AH = 0, B_AB = 16 * CS, B_A2 = 32 * CS, B_G0 = 48 * CS, B_G1 = 56 * CS, B_W0 = 64 * CS, B_W1 = B_W0 + 16384,
              B_SUM = B_W1 + 16384, B_BAR = B_SUM + 512;
constexpr int B_SMEM = B_BAR + 64;
static_assert(B_SMEM <= 232448, "backward kernel shared memory exceeds the 227 KB opt-in limit");

struct TtBwdArgs {
  TtLane ln;
  int B, ntile, nl, tiles_per_cta;
  TtLayer lay[4];
  const float* sgn_in[4];
  const float* sgn_out[4];
  float *g0, *g1;
  float keep[4];  // PLAIN mode: keep probability of the dropout site behind each layer (1 = none)
  long long lane_stride;  // ensemble members (blockIdx.z): bytes between their lanes
  int sign_stride;        // ensemble members: sign-tensor rows [B, C] between theirs (TtStep)
  int part_floats;
  int* status;
  long long* trace;
};

// gradient w.r.t. the layer OUTPUT (post-activation), 8 channels [n0, n0 + 8) of tile row `row`, and the ReLU gate
template <int MODE>
__device__ __forceinline__ void output_grad(const TtLane& ln, const TtLayer& L, int tile, int row, const RowInfo& ri, int n0,
                                            float (&d)[8]) {
#pragma unroll
  for (int j = 0; j < 8; ++j) d[j] = 0.f;
  if (!ri.live) return;
  if (L.out == OUT_FEAT) {
    const long long fa = feat_addr(ri.gw, ri.t, L.out_c0 + n0);
    float f[8], gr[8];
    unpack_h8(*reinterpret_cast<const uint4*>(ln.fimg + fa), f);
    unpack_b8(*reinterpret_cast<const uint4*>(ln.gfimg + fa), gr);
#pragma unroll
    for (int j = 0; j < 8; ++j) d[j] = f[j] > 0.f ? gr[j] : 0.f;
    return;
  }
  const long long ro = (long long)(ROW0 + row) * 16;
  float act[8], g[8];
  if (L.out != OUT_M1) {
    const int c = n0 >> 3;
    const unsigned char* ai = (L.out == OUT_T2 ? ln.t2 : ln.t3) + ((long long)tile * 8 + c) * CS + ro;
    const unsigned char* gi = ln.g[L.out == OUT_T2 ? 4 : 5] + ((long long)tile * 8 + c) * CS + ro;
    unpack_h8(*reinterpret_cast<const uint4*>(ai), act);
    unpack_b8(*reinterpret_cast<const uint4*>(gi), g);
#pragma unroll
    for (int j = 0; j < 8; ++j) d[j] = act[j] > 0.f ? g[j] : 0.f;
    return;
  }
  // module-1 output: three direct consumers + the pooled branch (route through MaxPool1d(3,1,1): first maximum wins)
  const long long co = ((long long)tile * 16 + L.out_c0 + (n0 >> 3)) * CS + ro;
  float m[5][8], gp[3][8];
#pragma unroll
  for (int q = 0; q < 5; ++q) unpack_h8(*reinterpret_cast<const uint4*>(ln.m1 + co + (q - 2) * 16), m[q]);
#pragma unroll
  for (int q = 0; q < 3; ++q) unpack_b8(*reinterpret_cast<const uint4*>(ln.g[3] + co + (q - 1) * 16), gp[q]);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    unpack_b8(*reinterpret_cast<const uint4*>(ln.g[k] + co), g);
#pragma unroll
    for (int j = 0; j < 8; ++j) d[j] += g[j];
  }
  const int t = ri.t;
#pragma unroll
  for (int dq = -1; dq <= 1; ++dq) {  // pooled position q = t + dq; does its window's first maximum sit at t?
    const int q = t + dq;
    if (q < 0 || q > 29) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      // window {q-1, q, q+1} clipped to [0, 29]; index into m[] is (position - t + 2)
      float best = -1.f;
      int arg = -9;
#pragma unroll
      for (int w = -1; w <= 1; ++w) {
        const int pos = q + w;
        if (pos < 0 || pos > 29) continue;
        const float v = m[pos - t + 2][j];
        if (v > best) { best = v; arg = pos; }
      }
      if (arg == t) d[j] += gp[dq + 1][j];
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) d[j] = m[2][j] > 0.f ? d[j] : 0.f;
}

template <int MODE>
__global__ void __launch_bounds__(NT, 1) tt_bwd_kernel(const TtBwdArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  const TtLayer& L = a.lay[blockIdx.y];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  long long* tr = (a.trace && blockIdx.x == 0 && blockIdx.z == 0 && tid == 0) ? a.trace + blockIdx.y * 16 : nullptr;
  const TtLane ln = member_lane(a.ln, a.lane_stride);
  if (tr) tr[0] = clock64();
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar_ld = sbase + B_BAR, bar_mma = bar_ld + 8;
  uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + B_BAR + 16);
  float* sums = reinterpret_cast<float*>(smem + B_SUM);  // [2][64] bias-gradient partial sums
  if (tid == 0) {
    mbar_init(bar_ld, 1);
    mbar_init(bar_mma, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc(smem_u32(tslot), 512);
  // zeros that must be there: the 4th k-chunk of an x input and the pad rows of the gradient images (they stay zero for the
  // whole kernel).  Chunks beyond KC are only read as M lanes >= KC * 8 of the weight-gradient MMAs, i.e. accumulator rows that
  // nobody reads back.
  for (int i = tid; i < CS / 16; i += NT) reinterpret_cast<uint4*>(smem + B_AH + 3 * CS)[i] = make_uint4(0, 0, 0, 0);
  if (tid < 64) {  // 16 gradient chunks (G0 | G1 are contiguous) x pad rows {0, 1, 130, 131}
    const int c = tid >> 2, r4 = tid & 3, pr = r4 < 2 ? r4 : 128 + r4;
    *reinterpret_cast<uint4*>(smem + B_G0 + c * CS + pr * 16) = make_uint4(0, 0, 0, 0);
  }
  if (tid < 128) sums[tid] = 0.f;
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tslot;
  if (tr) tr[8] = clock64();
  const bool has_dx = L.gdst >= 0;
  const int dxw = has_dx ? L.KC * 8 : 0;            // columns of one input-gradient accumulator
  const uint32_t t_dx0 = tmem, t_dx1 = tmem + dxw, t_dw0 = tmem + 2 * dxw, t_dw1 = t_dw0 + L.T * L.NP;
  const int ncopy = L.in <= IN_XP ? 3 : L.KC;
  const int img_bytes = L.T * L.tap_bytes;
  const int pad = (L.T - 1) >> 1;
  const int tile0 = blockIdx.x * a.tiles_per_cta, tile1 = min(a.ntile, tile0 + a.tiles_per_cta);
  uint32_t ph = 0;
  for (int tile = tile0; tile < tile1; ++tile) {
    if (tid == 0) {
      const bool first = tile == tile0;
      mbar_expect_tx(bar_ld, ncopy * CS + (first ? (MODE == TT_PLAIN ? 1 : 2) * img_bytes : 0));
      bulk_copy_chunked(sbase + (L.in == IN_M1P ? B_AB : B_AH), input_image(ln, L.in, tile), ncopy * CS, bar_ld);
      if (first) {
        bulk_copy_chunked(sbase + B_W0, ln.blob + L.w0b, img_bytes, bar_ld);
        if (MODE != TT_PLAIN) bulk_copy_chunked(sbase + B_W1, ln.blob + L.w1b, img_bytes, bar_ld);
      }
    }
    // ---- gradient operands (global reads only): G0 = d/d(pre-activation), G1 = d/d(variance) or d/d(perturbation);
    //      thread = row x chunk quarter
    const int row = (warp & 3) * 32 + lane, cq = warp >> 2;
    const RowInfo ri = row_info(ROW0 + row, tile, a.B);
    const float* rb = ln.rbuf + (long long)tile * RBUF_PER_TILE + L.roff_per_tile;
    const float* sout = member_ptr(a.sgn_out[blockIdx.y], (long long)a.sign_stride * a.B * L.N);
    for (int c = cq; c < L.NP / 8; c += 4) {
      float d[8], d1[8];
      output_grad<MODE>(ln, L, tile, row, ri, c * 8, d);
      if (MODE == TT_PLAIN && a.keep[blockIdx.y] < 1.0f) {  // dropout behind the ReLU: the stored activation a * m / keep gates, 1 / keep scales
        const float ik = 1.0f / a.keep[blockIdx.y];
#pragma unroll
        for (int j = 0; j < 8; ++j) d[j] *= ik;
      }
      if (tr && tile == tile0 && c == cq) tr[9] = clock64();
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int n = c * 8 + j;
        if (MODE == BRL_MODE_LRT) d1[j] = d[j] * rb[(long long)n * 128 + row];
        else if (MODE == BRL_MODE_FLIPOUT) d1[j] = (ri.live && n < L.N) ? d[j] * __ldg(sout + (long long)ri.gw * L.N + n) : 0.f;
        else d1[j] = 0.f;
      }
      *reinterpret_cast<uint4*>(smem + B_G0 + c * CS + (ROW0 + row) * 16) = pack_b8(d);
      if (MODE != TT_PLAIN) *reinterpret_cast<uint4*>(smem + B_G1 + c * CS + (ROW0 + row) * 16) = pack_b8(d1);
      if (tr && tile == tile0 && c == cq) tr[10] = clock64();
      {  // bias gradients: column sums over the tile's rows (lane 4 j holds channel j's)
        const float s0 = warp_sum8(d, lane), s1 = MODE == TT_PLAIN ? 0.f : warp_sum8(d1, lane);
        if ((lane & 3) == 0) { atomicAdd(&sums[c * 8 + (lane >> 2)], s0); atomicAdd(&sums[64 + c * 8 + (lane >> 2)], s1); }
      }
    }
    if (tr && tile == tile0) tr[1] = clock64();
    mbar_wait(bar_ld, ph, a.status, 42);
    if (tr && tile == tile0) tr[2] = clock64();
    if (L.in == IN_M1P) {
      pool_image(smem + B_AB, smem + B_AH, L.KC, tile, a.B, tid);
      __syncthreads();
    }
    second_operand<MODE, false>(smem + B_AH, smem + B_A2, smem + B_AB, L,
                                member_ptr(a.sgn_in[blockIdx.y], (long long)a.sign_stride * a.B * L.cin), tile, a.B, tid);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tr && tile == tile0) tr[3] = clock64();
    if (warp == 0) {
      tc_fence_after();
      if (elect_one()) {
        if (has_dx)  // D[row, c] += G[row - (tap - pad), n] * W[n, c, tap]: B = the weight image read MN-major
          for (int tap = 0; tap < L.T; ++tap)
            for (int ks = 0; ks < L.NP / 16; ++ks) {
              const uint32_t go = 2 * ks * CS + (ROW0 - (tap - pad)) * 16, wo = tap * L.tap_bytes + ks * 256;
              umma(t_dx0, umma_desc(sbase + B_G0 + go, CS, 128), umma_desc(sbase + B_W0 + wo, 128, L.NP * 16), tt_idesc(dxw, 1, 0, 1),
                   (tap | ks) != 0);
              if (MODE != TT_PLAIN)
                umma(t_dx1, umma_desc(sbase + B_G1 + go, CS, 128), umma_desc(sbase + B_W1 + wo, 128, L.NP * 16), tt_idesc(dxw, 1, 0, 1),
                     (tap | ks) != 0);
            }
        // D[c, n] += act[c, r + tap - pad] * G[n, r] over the tile's 128 rows: both operands MN-major, accumulated over the group
        for (int tap = 0; tap < L.T; ++tap)
          for (int ks = 0; ks < 8; ++ks) {
            const uint32_t ao = (ROW0 + tap - pad + 16 * ks) * 16, go = (ROW0 + 16 * ks) * 16;
            const uint32_t acc = (tile != tile0 || ks != 0) ? 1u : 0u;
            umma(t_dw0 + tap * L.NP, umma_desc(sbase + B_AB + ao, 128, CS), umma_desc(sbase + B_G0 + go, 128, CS), tt_idesc(L.NP, 1, 1, 1), acc);
            if (MODE != TT_PLAIN)
              umma(t_dw1 + tap * L.NP, umma_desc(sbase + B_A2 + ao, 128, CS), umma_desc(sbase + B_G1 + go, 128, CS), tt_idesc(L.NP, 1, 1, 1), acc);
          }
        umma_commit(bar_mma);
      }
      __syncwarp();
    }
    mbar_wait(bar_mma, ph, a.status, 43);
    tc_fence_after();
    ph ^= 1;
    if (tr && tile == tile0) tr[4] = clock64();
    if (has_dx) {  // ---- input gradient of this tile -> bf16 image (thread = row x column quarter)
      unsigned char* gi = member_ptr(a.ln.g[L.gdst], a.lane_stride) + (long long)tile * L.KC * CS;  // (ln.g[L.gdst]: a local-memory copy)
      const uint32_t la = tmem + ((uint32_t)((warp & 3) * 32) << 16);
      const float* sin_ = member_ptr(a.sgn_in[blockIdx.y], (long long)a.sign_stride * a.B * L.cin);
      for (int g = cq; g < dxw / 8; g += 4) {
        float v0[8], v1[8], o[8], av[8];
        tmem_ld8(la + g * 8, v0);
        if (MODE != TT_PLAIN) tmem_ld8(la + dxw + g * 8, v1);
        tmem_ld_wait();
        if (MODE == BRL_MODE_LRT) unpack_h8(*reinterpret_cast<const uint4*>(smem + B_AH + g * CS + (ROW0 + row) * 16), av);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float r = 0.f;
          if (ri.live) {
            if (MODE == BRL_MODE_LRT) r = fmaf(2.0f * av[j], v1[j], v0[j]);
            else if (MODE == BRL_MODE_FLIPOUT) {
              const int cr = real_ch(L.in, g * 8 + j);
              r = cr >= 0 ? fmaf(__ldg(sin_ + (long long)ri.gw * L.cin + cr), v1[j], v0[j]) : 0.f;
            } else r = v0[j];
          }
          o[j] = r;
        }
        *reinterpret_cast<uint4*>(gi + g * CS + (ROW0 + row) * 16) = pack_b8(o);
      }
      if (tid < 4) {
        const int pr = tid < 2 ? tid : 128 + tid;
        for (int c = 0; c < L.KC; ++c) *reinterpret_cast<uint4*>(gi + c * CS + pr * 16) = make_uint4(0, 0, 0, 0);
      }
    }
    tc_fence_before();
    __syncthreads();  // the next tile's copies / operand writes may overwrite what this tile's MMAs and epilogue read
    tc_fence_after();
    if (tr && tile == tile0) tr[5] = clock64();
  }
  // ---- weight gradients of the group: thread = TMEM lane = input channel of the image, (tap, 8 output channels) items spread
  //      over the column quarters
  if (tile0 < tile1) {
    const int ch = (warp & 3) * 32 + lane, cq = warp >> 2;
    const int CH = L.KC * 8;
    float* part = ln.part + (long long)blockIdx.x * a.part_floats + L.poff;
    const uint32_t la = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const int ng = L.NP / 8;
    for (int it = cq; it < L.T * ng; it += 4) {
      const int tap = it / ng, g = it - tap * ng;
      float v0[8], v1[8];
      tmem_ld8(la + 2 * dxw + tap * L.NP + g * 8, v0);
      if (MODE != TT_PLAIN) tmem_ld8(la + 2 * dxw + (L.T + tap) * L.NP + g * 8, v1);
      tmem_ld_wait();
      // plain, coalesced stores (lanes = consecutive image channels) into this group's block of partials; tt_reduce_kernel sums
      // the groups -- 64 CTAs adding to the same 33 k addresses with atomics cost 8 - 13 us per level
      if (ch < CH) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int n = g * 8 + j;
          if (n < L.N) {
            part[((long long)n * L.T + tap) * CH + ch] = v0[j];
            if (MODE != TT_PLAIN) part[(long long)L.N * L.T * CH + ((long long)n * L.T + tap) * CH + ch] = v1[j];
          }
        }
      }
    }
    if (tid < 128) part[2ll * L.N * L.T * CH + tid] = sums[tid];
  }
  if (tr) tr[6] = clock64();
  tc_fence_before();
  __syncthreads();
  if (tr) tr[7] = clock64();
  if (warp == 0) tmem_dealloc(tmem, 512);
}


// ------------------------------------------------------------------------------------------------
// fc layer (2400 -> 64) on the tensor pipe: forward (split-K partial sums for the per-layer engine's split-K epilogue, which
// applies bias / eps * sqrt(var) / sign flips / ReLU exactly as for the fp32 kernels), input gradient, weight gradient
// ------------------------------------------------------------------------------------------------
struct TtFcPackArgs {
  int mode;
  const float *mu, *second;
  long long w_off;
  unsigned char* blob;  // w0h | w0b | w1b | w1h, FC_WIMG bytes each
  long long P, lane_stride;  // ensemble members (blockIdx.z): parameter / lane strides
};
__global__ void tt_pack_fc_kernel(const TtFcPackArgs a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 64 * 2400) return;
  const int n = i / 2400, kp = i - n * 2400, t = kp / 80, c = kp - t * 80;
  const long long wi = a.w_off + (long long)n * 2400 + c * 30 + t;
  const float m = a.mu[wi + a.P * blockIdx.z], v = a.second[wi + a.P * blockIdx.z];
  const float s = a.mode == BRL_MODE_LRT ? v * v : a.mode == BRL_MODE_FLIPOUT ? v - m : 0.f;
  const long long o = a.lane_stride * blockIdx.z + (kp >> 3) * 1024 + n * 16 + (kp & 7) * 2;
  *reinterpret_cast<__half*>(a.blob + o) = __float2half_rn(m);
  *reinterpret_cast<__nv_bfloat16*>(a.blob + FC_WIMG + o) = __float2bfloat16_rn(m);
  *reinterpret_cast<__nv_bfloat16*>(a.blob + 2 * FC_WIMG + o) = __float2bfloat16_rn(s);
  *reinterpret_cast<__half*>(a.blob + 3 * FC_WIMG + o) = __float2half_rn(s);
}

constexpr int FF_A = 0, FF_A2 = FC_KCS * FC_CHUNK, FF_W0 = 2 * FC_KCS * FC_CHUNK, FF_W1 = FF_W0 + FC_KCS * 1024, FF_BAR = FF_W1 + FC_KCS * 1024;
constexpr int FF_SMEM = FF_BAR + 64;
struct TtFcFwdArgs {
  TtLane ln;
  int B, mode;
  float* part;  // [2][B][64] fp32, zeroed: mean-path and second-path sums (brl_gemm.cu split-K scratch layout)
  long long lane_stride, part_stride;  // ensemble members (blockIdx.z): bytes between their lanes, floats between their `part`
  int* status;
};
__global__ void __launch_bounds__(256, 1) tt_fc_fwd_kernel(const TtFcFwdArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int mt = blockIdx.x, ks = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem), bar_ld = sbase + FF_BAR, bar_mma = bar_ld + 8;
  uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + FF_BAR + 16);
  const TtLane ln = member_lane(a.ln, a.lane_stride);
  float* part = a.part + a.part_stride * blockIdx.z;
  if (tid == 0) {
    mbar_init(bar_ld, 1);
    mbar_init(bar_mma, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc(smem_u32(tslot), 128);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tslot;
  if (tid == 0) {
    const long long ao = ((long long)mt * FC_KC + ks * FC_KCS) * FC_CHUNK;
    const bool dual = a.mode == BRL_MODE_LRT || a.mode == BRL_MODE_FLIPOUT;
    mbar_expect_tx(bar_ld, (dual ? 2 : 1) * (FC_KCS * FC_CHUNK + FC_KCS * 1024));
    bulk_copy_chunked(sbase + FF_A, ln.fimg + ao, FC_KCS * FC_CHUNK, bar_ld);
    bulk_copy_chunked(sbase + FF_W0, ln.fcblob + (long long)ks * FC_KCS * 1024, FC_KCS * 1024, bar_ld);
    if (dual) bulk_copy_chunked(sbase + FF_A2, ln.f2img + ao, FC_KCS * FC_CHUNK, bar_ld);
    if (dual) bulk_copy_chunked(sbase + FF_W1, ln.fcblob + (a.mode == BRL_MODE_LRT ? 2 : 3) * (long long)FC_WIMG + (long long)ks * FC_KCS * 1024, FC_KCS * 1024, bar_ld);
  }
  mbar_wait(bar_ld, 0, a.status, 44);
  if (warp == 0) {
    tc_fence_after();
    if (elect_one()) {
      for (int k = 0; k < FC_KCS / 2; ++k) {
        umma(tmem, umma_desc(sbase + FF_A + 2 * k * FC_CHUNK, FC_CHUNK, 128), umma_desc(sbase + FF_W0 + 2 * k * 1024, 1024, 128),
             tt_idesc(64, 0, 0, 0), k != 0);
        if (a.mode == BRL_MODE_LRT || a.mode == BRL_MODE_FLIPOUT)
          umma(tmem + 64, umma_desc(sbase + FF_A2 + 2 * k * FC_CHUNK, FC_CHUNK, 128), umma_desc(sbase + FF_W1 + 2 * k * 1024, 1024, 128),
               tt_idesc(64, a.mode == BRL_MODE_LRT ? 1 : 0, 0, 0), k != 0);
      }
      umma_commit(bar_mma);
    }
    __syncwarp();
  }
  mbar_wait(bar_mma, 0, a.status, 45);
  tc_fence_after();
  const int m = mt * 128 + (warp & 3) * 32 + lane, half = warp >> 2;
  const uint32_t la = tmem + ((uint32_t)((warp & 3) * 32) << 16);
#pragma unroll 1
  for (int g = 0; g < 2; ++g) {
    const bool dual = a.mode == BRL_MODE_LRT || a.mode == BRL_MODE_FLIPOUT;
    float v0[16], v1[16];
    tmem_ld16(la + half * 32 + g * 16, v0);
    if (dual) tmem_ld16(la + 64 + half * 32 + g * 16, v1);
    tmem_ld_wait();
    if (m < a.B) {
      float* p0 = part + (long long)m * 64 + half * 32 + g * 16;
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        atomicAdd(p0 + j, v0[j]);
        if (dual) atomicAdd(p0 + (long long)a.B * 64 + j, v1[j]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 128);
}

// gradient operands of the fc layer: compact fp32 [B, 64] (bwd_act_kernel) -> bf16 K-major image [8 chunks][128 windows][16 B]
__device__ __forceinline__ void fc_grad_image(const float* __restrict__ d, unsigned char* img, int mt, int B, int tid, int nthreads) {
  for (int i = tid; i < 128 * 8; i += nthreads) {
    const int r = i & 127, c = i >> 7, m = mt * 128 + r;
    float v[8];
    if (m < B) {
      const float4 lo = *reinterpret_cast<const float4*>(d + (long long)m * 64 + c * 8), hi = *reinterpret_cast<const float4*>(d + (long long)m * 64 + c * 8 + 4);
      v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w; v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = 0.f;
    }
    *reinterpret_cast<uint4*>(img + c * FC_CHUNK + r * 16) = pack_b8(v);
  }
}

constexpr int FX_G0 = 0, FX_G1 = 8 * FC_CHUNK, FX_W0 = 16 * FC_CHUNK, FX_W1 = FX_W0 + FC_NCS * 1024, FX_BAR = FX_W1 + FC_NCS * 1024;
constexpr int FX_SMEM = FX_BAR + 64;
struct TtFcBwdArgs {
  TtLane ln;
  int B, nmt, mode;
  const float *dpre, *dsec;  // [B, 64] fp32
  const float* sgn_in;       // Flipout [B, 2400]
  float *g0, *g1;
  long long w_off, b_off;
  long long P, lane_stride;  // ensemble members (blockIdx.z): parameter / lane strides; dpre / dsec [members][B][64]
  int* status;
};
// the arguments as ensemble member blockIdx.z sees them
__device__ __forceinline__ TtFcBwdArgs member_fc(TtFcBwdArgs a) {
  a.ln = member_lane(a.ln, a.lane_stride);
  a.dpre = member_ptr(a.dpre, 64ll * a.B);
  a.dsec = member_ptr(a.dsec, 64ll * a.B);
  a.g0 = member_ptr(a.g0, a.P);
  a.g1 = member_ptr(a.g1, a.P);
  return a;
}
// d/d(features)[m, k'] = dpre[m, :] * W0[:, k'] + {2 f, s_in}[m, k'] * (dsec[m, :] * W1[:, k'])  -> bf16 image for the level kernels
template <int MODE>
__global__ void __launch_bounds__(256, 1) tt_fc_dx_kernel(const TtFcBwdArgs a_) {
  extern __shared__ __align__(128) unsigned char smem[];
  const TtFcBwdArgs a = member_fc(a_);
  const int mt = blockIdx.x, ns = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem), bar_ld = sbase + FX_BAR, bar_mma = bar_ld + 8;
  uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + FX_BAR + 16);
  if (tid == 0) {
    mbar_init(bar_ld, 1);
    mbar_init(bar_mma, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc(smem_u32(tslot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tslot;
  if (tid == 0) {
    mbar_expect_tx(bar_ld, (MODE == TT_PLAIN ? 1 : 2) * FC_NCS * 1024);
    bulk_copy_chunked(sbase + FX_W0, a.ln.fcblob + FC_WIMG + (long long)ns * FC_NCS * 1024, FC_NCS * 1024, bar_ld);
    if (MODE != TT_PLAIN) bulk_copy_chunked(sbase + FX_W1, a.ln.fcblob + 2 * FC_WIMG + (long long)ns * FC_NCS * 1024, FC_NCS * 1024, bar_ld);
  }
  fc_grad_image(a.dpre, smem + FX_G0, mt, a.B, tid, 256);
  if (MODE != TT_PLAIN) fc_grad_image(a.dsec, smem + FX_G1, mt, a.B, tid, 256);
  mbar_wait(bar_ld, 0, a.status, 46);
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    if (elect_one()) {
      for (int k = 0; k < 4; ++k) {  // K = 64 output units; B = the weight image read MN-major: [N' = FC_NCS * 8 features][K' = 16 units]
        umma(tmem, umma_desc(sbase + FX_G0 + 2 * k * FC_CHUNK, FC_CHUNK, 128), umma_desc(sbase + FX_W0 + k * 256, 128, 1024),
             tt_idesc(FC_NCS * 8, 1, 0, 1), k != 0);
        if (MODE != TT_PLAIN)
          umma(tmem + 256, umma_desc(sbase + FX_G1 + 2 * k * FC_CHUNK, FC_CHUNK, 128), umma_desc(sbase + FX_W1 + k * 256, 128, 1024),
               tt_idesc(FC_NCS * 8, 1, 0, 1), k != 0);
      }
      umma_commit(bar_mma);
    }
    __syncwarp();
  }
  mbar_wait(bar_mma, 0, a.status, 47);
  tc_fence_after();
  const int r = (warp & 3) * 32 + lane, gw = mt * 128 + r, half = warp >> 2;
  const uint32_t la = tmem + ((uint32_t)((warp & 3) * 32) << 16);
#pragma unroll 1
  for (int g = half; g < FC_NCS; g += 2) {
    float v0[8], v1[8], o[8], f[8];
    tmem_ld8(la + g * 8, v0);
    if (MODE != TT_PLAIN) tmem_ld8(la + 256 + g * 8, v1);
    const int kc = ns * FC_NCS + g, t = kc / 10, c0 = (kc - t * 10) * 8;
    const long long fa = ((long long)mt * FC_KC + kc) * FC_CHUNK + r * 16;
    // LRT: the factor is 2 f.  Flipout: s_in, read back as the sign of the perturbation operand f * s_in (f >= 0 behind the ReLU;
    // where f == 0 the consumer masks this gradient anyway) -- one coalesced 16-byte load instead of eight strided sign loads
    if (MODE != TT_PLAIN) unpack_h8(*reinterpret_cast<const uint4*>((MODE == BRL_MODE_LRT ? a.ln.fimg : a.ln.f2img) + fa), f);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (MODE == TT_PLAIN) { o[j] = gw < a.B ? v0[j] : 0.f; continue; }
      const float mul = MODE == BRL_MODE_LRT ? 2.0f * f[j] : (signbit(f[j]) ? -1.0f : 1.0f);
      o[j] = gw < a.B ? fmaf(mul, v1[j], v0[j]) : 0.f;
    }
    *reinterpret_cast<uint4*>(a.ln.gfimg + fa) = pack_b8(o);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512);
}

constexpr int FW_A = 0, FW_A2 = 16 * FC_CHUNK, FW_G0 = 32 * FC_CHUNK, FW_G1 = 40 * FC_CHUNK, FW_BAR = 48 * FC_CHUNK;
constexpr int FW_SMEM = FW_BAR + 64;
// weight gradient: D[k', n] = sum_m F[m, k'] * dpre[m, n] (and the second path), M = 128 features per CTA, K = all windows
template <int MODE>
__global__ void __launch_bounds__(256, 1) tt_fc_dw_kernel(const TtFcBwdArgs a_) {
  extern __shared__ __align__(128) unsigned char smem[];
  const TtFcBwdArgs a = member_fc(a_);
  const int kt = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem), bar_ld = sbase + FW_BAR, bar_mma = bar_ld + 8;
  uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + FW_BAR + 16);
  if (tid == 0) {
    mbar_init(bar_ld, 1);
    mbar_init(bar_mma, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc(smem_u32(tslot), 128);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tslot;
  const int nch = min(16, FC_KC - kt * 16);  // the last tile holds 12 chunks: features beyond 2400 are accumulator rows nobody reads
  uint32_t ph = 0;
  for (int mt = 0; mt < a.nmt; ++mt) {
    if (tid == 0) {
      const long long ao = ((long long)mt * FC_KC + kt * 16) * FC_CHUNK;
      mbar_expect_tx(bar_ld, (MODE == TT_PLAIN ? 1 : 2) * nch * FC_CHUNK);
      bulk_copy_chunked(sbase + FW_A, a.ln.fbimg + ao, nch * FC_CHUNK, bar_ld);
      if (MODE != TT_PLAIN) bulk_copy_chunked(sbase + FW_A2, (MODE == BRL_MODE_LRT ? a.ln.f2img : a.ln.f2bimg) + ao, nch * FC_CHUNK, bar_ld);
    }
    fc_grad_image(a.dpre, smem + FW_G0, mt, a.B, tid, 256);
    if (MODE != TT_PLAIN) fc_grad_image(a.dsec, smem + FW_G1, mt, a.B, tid, 256);
    mbar_wait(bar_ld, ph, a.status, 48);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
      if (elect_one()) {
        for (int k = 0; k < 8; ++k) {  // 16 windows per k-step; both operands MN-major
          const uint32_t acc = (mt | k) != 0;
          umma(tmem, umma_desc(sbase + FW_A + k * 256, 128, FC_CHUNK), umma_desc(sbase + FW_G0 + k * 256, 128, FC_CHUNK),
               tt_idesc(64, 1, 1, 1), acc);
          if (MODE != TT_PLAIN)
            umma(tmem + 64, umma_desc(sbase + FW_A2 + k * 256, 128, FC_CHUNK), umma_desc(sbase + FW_G1 + k * 256, 128, FC_CHUNK),
                 tt_idesc(64, 1, 1, 1), acc);
        }
        umma_commit(bar_mma);
      }
      __syncwarp();
    }
    mbar_wait(bar_mma, ph, a.status, 49);
    tc_fence_after();
    ph ^= 1;
    __syncthreads();
  }
  const int kp = kt * 128 + (warp & 3) * 32 + lane, half = warp >> 2;
  const uint32_t la = tmem + ((uint32_t)((warp & 3) * 32) << 16);
#pragma unroll 1
  for (int g = 0; g < 2; ++g) {
    float v0[16], v1[16];
    tmem_ld16(la + half * 32 + g * 16, v0);
    if (MODE != TT_PLAIN) tmem_ld16(la + 64 + half * 32 + g * 16, v1);
    tmem_ld_wait();
    if (kp < 2400) {
      const int t = kp / 80, c = kp - t * 80;
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const long long wi = a.w_off + (long long)(half * 32 + g * 16 + j) * 2400 + c * 30 + t;
        a.g0[wi] = v0[j];
        if (MODE != TT_PLAIN) a.g1[wi] = v1[j];
      }
    }
  }
  {  // bias gradients: column sums of the compact gradient tensors, a slice of windows per CTA and per thread group
    const int n = tid & 63, q = tid >> 6, nsl = gridDim.x * 4, sl = blockIdx.x * 4 + q;
    const int per = (a.B + nsl - 1) / nsl, m0 = sl * per, m1 = min(a.B, m0 + per);
    float s0 = 0.f, s1 = 0.f;
#pragma unroll 4
    for (int m = m0; m < m1; ++m) {
      s0 += a.dpre[(long long)m * 64 + n];
      if (MODE != TT_PLAIN) s1 += a.dsec[(long long)m * 64 + n];
    }
    if (m0 < m1) {
      atomicAdd(a.g0 + a.b_off + n, s0);
      if (MODE != TT_PLAIN) atomicAdd(a.g1 + a.b_off + n, MODE == BRL_MODE_LRT ? s1 : s0);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 128);
}


// ------------------------------------------------------------------------------------------------
// tail of the net in ONE launch: fc epilogue (bias, eps * sqrt(var) / sign flips, ReLU) -> head 64 -> 2 (dual) -> softplus +
// Threshold(1e-9) -> ELBO likelihood (second softplus, bayesian.py:73-76) and its gradient -> head backward (input and weight
// gradients) -> activation backward of the fc layer (the compact dpre / dsec tensors of tt_fc_backward).  It replaces eight
// per-layer launches (split-K epilogue, head GEMM, NLL, two activation-backward, head dX / dW) of 3 - 11 us each; the arithmetic
// is that of brl_gemm_epi.cuh / nll_elbo_kernel / bwd_act_kernel, one warp per window, lane = hidden units {lane, lane + 32}.
// HW = width of the hidden layer in front of the head: 64 (Inception fc layer), 32 (Linear layer 3, lane = hidden unit lane),
// 320 (Conv-D3: `part` holds the pooled, activated conv3 features [B, 320] as they are -- no fc epilogue -- and `dpre` receives
// their gradient).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double tt_block_sum(double v) {  // valid in thread 0
  __shared__ double red[32];
  __syncthreads();
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x < 32) {
    v = threadIdx.x < (blockDim.x + 31) / 32 ? red[threadIdx.x] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  }
  return v;
}
struct TtTailArgs {
  int B, mode, compute_grads;
  const float* part;           // [2][B][HW] fc partial sums (mean path, second path)
  const float *fc_b0, *fc_b1;  // LRT: mu_b, sigma_b of the fc layer; Flipout: fc_b0 = sampled bias
  const float *hw0, *hw1;      // head weights [2][HW]: LRT mu, sigma; Flipout mu, sampled W
  const float *hb0, *hb1;      // head bias [2]:      LRT mu_b, sigma_b; Flipout hb0 = sampled bias
  NoiseRef eps_fc, eps_head;   // LRT
  const float *sout_fc, *sin_head, *sout_head;  // Flipout [B,HW], [B,HW], [B,2]
  const float* y;
  float gscale;
  double* acc;                 // [0] += nll, [1] += squared error
  float* out;                  // [B,2]
  float *dpre, *dsec;          // [B,HW] compact gradients of the fc layer's pre-activation / second path
  float *g0, *g1;              // flat gradient accumulators (head layer: atomics)
  long long hw_off, hb_off;
  // PLAIN mode (one contraction: HNN / MC-dropout step, weight-sampling ELBO): fc_b0 / hw0 / hb0 are the weights in use
  int loss_kind;               // 0: ELBO likelihood (second softplus, sums in acc); 1: F.gaussian_nll_loss (frequentist.py:39-48, means in acc)
  float keep_fc;               // keep probability of the dropout site behind the fc layer (1 = none)
  NoiseRef drop_fc;            // its masks: injected [B, HW] or Philox
  long long P, part_stride;    // ensemble members (blockIdx.z): floats between their parameters / gradients and their `part`
  int noise_stride, sign_stride, acc_stride;  // ... MC samples / sign rows [B, C] / accumulator doubles between theirs
};
// the arguments as ensemble member blockIdx.z sees them (y, dpre, dsec: [members][B][...]; out: [members][noise_stride][B][2];
// acc: [members][acc_stride])
template <int HW>
__device__ __forceinline__ TtTailArgs member_tail(TtTailArgs a) {
  a.part = member_ptr(a.part, a.part_stride);
  a.fc_b0 = member_ptr(a.fc_b0, a.P); a.fc_b1 = member_ptr(a.fc_b1, a.P);
  a.hw0 = member_ptr(a.hw0, a.P); a.hw1 = member_ptr(a.hw1, a.P);
  a.hb0 = member_ptr(a.hb0, a.P); a.hb1 = member_ptr(a.hb1, a.P);
  a.y = member_ptr(a.y, (long long)a.B);
  a.acc = member_ptr(a.acc, (long long)a.acc_stride);
  a.out = member_ptr(a.out, 2ll * a.noise_stride * a.B);
  a.dpre = member_ptr(a.dpre, (long long)HW * a.B); a.dsec = member_ptr(a.dsec, (long long)HW * a.B);
  a.g0 = member_ptr(a.g0, a.P); a.g1 = member_ptr(a.g1, a.P);
  a.drop_fc = member_noise(a.drop_fc, HW, a.B, a.noise_stride);
  a.eps_fc = member_noise(a.eps_fc, HW, a.B, a.noise_stride);
  a.eps_head = member_noise(a.eps_head, 2, a.B, a.noise_stride);
  const long long sr = (long long)a.sign_stride * a.B;
  a.sout_fc = member_ptr(a.sout_fc, sr * HW); a.sin_head = member_ptr(a.sin_head, sr * HW); a.sout_head = member_ptr(a.sout_head, sr * 2);
  return a;
}
template <int MODE, int HW>
__global__ void __launch_bounds__(256) tt_tail_kernel(const TtTailArgs a_) {
  const TtTailArgs a = member_tail<HW>(a_);
  __shared__ float sg[2][2][HW + 1];  // [path][output][hidden unit | bias] head weight-gradient partials of the CTA
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < 2 * 2 * (HW + 1); i += 256) (&sg[0][0][0])[i] = 0.f;
  __syncthreads();
  constexpr int U = HW / 32;  // hidden units per lane
  constexpr bool FEAT = HW == 320;
  float w0[2][U], w1[2][U];  // head weights of this lane's hidden units: [output][unit]
#pragma unroll
  for (int o = 0; o < 2; ++o)
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int k = lane + 32 * u;
      const float m = a.hw0[o * HW + k], v = MODE == TT_PLAIN ? 0.f : a.hw1[o * HW + k];
      w0[o][u] = m;
      w1[o][u] = MODE == BRL_MODE_LRT ? v * v : v - m;
    }
  float gw0[2][U] = {}, gw1[2][U] = {}, gb0[2] = {0.f, 0.f}, gb1[2] = {0.f, 0.f};
  double nll = 0.0, se = 0.0;
  const int nwarps = gridDim.x * 8;
  for (int m = blockIdx.x * 8 + warp; m < a.B; m += nwarps) {
    // ---- fc epilogue
    float h[U], sd[U], ef[U], sgn_in[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int k = lane + 32 * u;
      if (FEAT) {
        h[u] = a.part[(long long)m * HW + k];
        sd[u] = ef[u] = 0.f;
        sgn_in[u] = MODE == BRL_MODE_FLIPOUT ? a.sin_head[(long long)m * HW + k] : 0.f;
        continue;
      }
      const float a0 = a.part[(long long)m * HW + k], a1 = MODE == TT_PLAIN ? 0.f : a.part[((long long)a.B + m) * HW + k];
      float pre;
      if (MODE == TT_PLAIN) {
        pre = a0 + a.fc_b0[k];
        sd[u] = ef[u] = sgn_in[u] = 0.f;
      } else if (MODE == BRL_MODE_LRT) {
        const float sb = a.fc_b1[k];
        float var = fmaf(sb, sb, a1);
        if (var < 0.f) var += fabsf(var) + 1e-6f;
        sd[u] = sqrtf(var);
        ef[u] = gnoise_normal(a.eps_fc, 0, m, a.B, HW, k);
        pre = fmaf(sd[u], ef[u], a0 + a.fc_b0[k]);
        sgn_in[u] = 0.f;
      } else {
        ef[u] = a.sout_fc[(long long)m * HW + k];
        pre = a0 + a1 * ef[u] + a.fc_b0[k];
        sd[u] = 0.f;
        sgn_in[u] = a.sin_head[(long long)m * HW + k];
      }
      h[u] = fmaxf(pre, 0.f);
      if (MODE == TT_PLAIN && a.keep_fc < 1.0f) {  // dropout behind the fc layer's ReLU (inception.py:204-206)
        bool kp;
        if (a.drop_fc.ptr) kp = a.drop_fc.ptr[(long long)m * HW + k] != 0.f;
        else {
          const NoiseKey dk = noise_key(a.drop_fc);
          kp = philox_keep(dk.seed, a.drop_fc.kind, a.drop_fc.site, dk.sample0, dk.window0 + m, HW, 0, k, a.keep_fc);
        }
        h[u] = kp ? h[u] / a.keep_fc : 0.f;
      }
    }
    // ---- head: two outputs x two paths, reduced over the HW hidden units
    float p0[2], p1[2];
#pragma unroll
    for (int o = 0; o < 2; ++o) {
      float s0 = 0.f, s1 = 0.f;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        s0 = fmaf(h[u], w0[o][u], s0);
        if (MODE != TT_PLAIN) s1 = fmaf(MODE == BRL_MODE_LRT ? h[u] * h[u] : h[u] * sgn_in[u], w1[o][u], s1);
      }
      p0[o] = warp_sum(s0);
      p1[o] = MODE == TT_PLAIN ? 0.f : warp_sum(s1);
    }
    float outv[2], sdo[2], eo[2];
#pragma unroll
    for (int o = 0; o < 2; ++o) {
      float v;
      if (MODE == TT_PLAIN) {
        v = p0[o] + a.hb0[o];
        sdo[o] = eo[o] = 0.f;
      } else if (MODE == BRL_MODE_LRT) {
        const float sb = a.hb1[o];
        float var = fmaf(sb, sb, p1[o]);
        if (var < 0.f) var += fabsf(var) + 1e-6f;
        sdo[o] = sqrtf(var);
        eo[o] = gnoise_normal(a.eps_head, 0, m, a.B, 2, o);
        v = fmaf(sdo[o], eo[o], p0[o] + a.hb0[o]);
      } else {
        eo[o] = a.sout_head[(long long)m * 2 + o];
        sdo[o] = 0.f;
        v = p0[o] + p1[o] * eo[o] + a.hb0[o];
      }
      v = v > 20.0f ? v : log1pf(expf(v));
      outv[o] = v > 1e-9f ? v : 1e-9f;
    }
    if (lane == 0) *reinterpret_cast<float2*>(a.out + 2ll * m) = make_float2(outv[0], outv[1]);
    // ---- likelihood (SURVEY A.6) and its gradient w.r.t. the two outputs
    const float loc = outv[0], sc = outv[1];
    float go[2];
    if (MODE == TT_PLAIN && a.loss_kind == 1) {  // F.gaussian_nll_loss(loc, y, scale^2): eps clamp 1e-6 on the variance (gradient
                                                 // through the clamped value, as nll_hnn_kernel), mean reduction
      const float var = fmaxf(sc * sc, 1e-6f), dl = loc - a.y[m], invB = 1.0f / (float)a.B;
      if (lane == 0) {
        nll += 0.5 * ((double)logf(var) + (double)dl * dl / var);
        se += (double)dl * dl;
      }
      go[0] = dl / var * invB;
      go[1] = 0.5f * (1.0f / var - dl * dl / (var * var)) * 2.0f * sc * invB;
    } else {
      const float s = sc > 20.0f ? sc : log1pf(expf(sc));
      const float dy = a.y[m] - loc, r = dy / s;
      if (lane == 0) {
        nll += 0.5 * (double)r * r + (double)logf(s) + 0.9189385332046727;
        se += (double)dy * dy;
      }
      const float sig = sc > 20.0f ? 1.0f : 1.0f / (1.0f + expf(-sc));
      go[0] = -r / s * a.gscale;
      go[1] = (1.0f - r * r) / s * sig * a.gscale;
    }
    if (!a.compute_grads) continue;
    // ---- head backward
    float d[2], d1[2];
#pragma unroll
    for (int o = 0; o < 2; ++o) {
      d[o] = outv[o] > 1e-9f ? go[o] * -expm1f(-outv[o]) : 0.f;
      d1[o] = MODE == TT_PLAIN ? 0.f : MODE == BRL_MODE_LRT ? (sdo[o] > 0.f ? d[o] * eo[o] / (2.0f * sdo[o]) : 0.f) : d[o] * eo[o];
      gb0[o] += d[o];
      gb1[o] += MODE == BRL_MODE_LRT ? d1[o] : d[o];
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int k = lane + 32 * u;
      const float x1 = MODE == BRL_MODE_LRT ? h[u] * h[u] : h[u] * sgn_in[u];
      float dh0 = 0.f, dh1 = 0.f;
#pragma unroll
      for (int o = 0; o < 2; ++o) {
        gw0[o][u] = fmaf(d[o], h[u], gw0[o][u]);
        gw1[o][u] = fmaf(d1[o], x1, gw1[o][u]);
        dh0 = fmaf(d[o], w0[o][u], dh0);
        dh1 = fmaf(d1[o], w1[o][u], dh1);
      }
      const float dh = MODE == TT_PLAIN ? dh0 : MODE == BRL_MODE_LRT ? fmaf(2.0f * h[u], dh1, dh0) : fmaf(sgn_in[u], dh1, dh0);
      if (FEAT) {
        a.dpre[(long long)m * HW + k] = dh;
        continue;
      }
      // ---- activation backward of the fc layer (with dropout the stored activation is a * m / keep: it gates, 1 / keep scales)
      const float dp = h[u] > 0.f ? (MODE == TT_PLAIN ? dh / a.keep_fc : dh) : 0.f;
      a.dpre[(long long)m * HW + k] = dp;
      if (MODE != TT_PLAIN) a.dsec[(long long)m * HW + k] = MODE == BRL_MODE_LRT ? (sd[u] > 0.f ? dp * ef[u] / (2.0f * sd[u]) : 0.f) : dp * ef[u];
    }
  }
  // ---- reductions: likelihood sums (lane 0 of every warp holds its windows'), head weight gradients
  nll = tt_block_sum(nll);
  se = tt_block_sum(se);
  if (tid == 0) {
    const double sc_ = (MODE == TT_PLAIN && a.loss_kind == 1) ? 1.0 / (double)a.B : 1.0;  // HNN: means (nll_hnn_kernel)
    atomicAdd(a.acc + 0, nll * sc_);
    atomicAdd(a.acc + 1, se * sc_);
  }
  if (!a.compute_grads) return;
#pragma unroll
  for (int o = 0; o < 2; ++o) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      atomicAdd(&sg[0][o][lane + 32 * u], gw0[o][u]);
      atomicAdd(&sg[1][o][lane + 32 * u], gw1[o][u]);
    }
    if (lane == 0) {  // d[o] is warp-uniform: one lane carries the bias gradient
      atomicAdd(&sg[0][o][HW], gb0[o]);
      atomicAdd(&sg[1][o][HW], gb1[o]);
    }
  }
  __syncthreads();
  for (int i = tid; i < (MODE == TT_PLAIN ? 1 : 2) * 2 * (HW + 1); i += 256) {
    const int path = i / (2 * (HW + 1)), r = i - path * 2 * (HW + 1), o = r / (HW + 1), k = r - o * (HW + 1);
    float* g = path ? a.g1 : a.g0;
    atomicAdd(g + (k < HW ? a.hw_off + o * HW + k : a.hb_off + o), sg[path][o][k]);
  }
}

// weight / bias gradients of the ten conv layers: sum of the groups' partial blocks -> flat gradient accumulators
struct TtReduceArgs {
  TtLayer L[TT_LAYERS];
  int start[TT_LAYERS + 1];  // work items per layer: N * T * CH weights + N biases
  int ngroups[TT_LAYERS];
  int part_floats, mode;
  const float* part;
  float *g0, *g1;
  long long P, lane_stride;  // ensemble members (blockIdx.z): parameter / lane strides
};
constexpr int RED_SPLIT = 8;  // group ranges per output: blockIdx.y; each thread keeps <= 2 x 8 independent loads in flight
__global__ void tt_reduce_kernel(const TtReduceArgs a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.start[TT_LAYERS]) return;
  int li = 0;
  while (i >= a.start[li + 1]) ++li;
  const TtLayer& l = a.L[li];
  const int CH = l.KC * 8, nw = l.N * l.T * CH;
  const int j = i - a.start[li];
  const int per = (a.ngroups[li] + RED_SPLIT - 1) / RED_SPLIT;
  const int g_lo = blockIdx.y * per, g_hi = min(a.ngroups[li], g_lo + per);
  if (g_lo >= g_hi) return;
  const float* p = reinterpret_cast<const float*>(reinterpret_cast<const unsigned char*>(a.part) + a.lane_stride * blockIdx.z) + l.poff;
  float* g0 = a.g0 + a.P * blockIdx.z;
  float* g1 = member_ptr(a.g1, a.P);
  const bool dual = a.mode == BRL_MODE_LRT || a.mode == BRL_MODE_FLIPOUT;
  float s0 = 0.f, s1 = 0.f;
  if (j < nw) {
    const int ch = j % CH, cr = real_ch(l.in, ch);
    if (cr < 0) return;
#pragma unroll 8
    for (int gidx = g_lo; gidx < g_hi; ++gidx) {
      s0 += p[(long long)gidx * a.part_floats + j];
      if (dual) s1 += p[(long long)gidx * a.part_floats + nw + j];
    }
    const int nt_ = j / CH, n = nt_ / l.T, tap = nt_ - n * l.T;
    const long long wi = l.w_off + ((long long)n * l.cin + cr) * l.T + tap;
    atomicAdd(g0 + wi, s0);
    if (dual) atomicAdd(g1 + wi, s1);
  } else {
    const int n = j - nw;
#pragma unroll 8
    for (int gidx = g_lo; gidx < g_hi; ++gidx) {
      s0 += p[(long long)gidx * a.part_floats + 2ll * nw + n];
      if (dual) s1 += p[(long long)gidx * a.part_floats + 2ll * nw + 64 + n];
    }
    atomicAdd(g0 + l.b_off + n, s0);
    if (dual) atomicAdd(g1 + l.b_off + n, a.mode == BRL_MODE_LRT ? s1 : s0);  // Flipout: the sampled bias (brl_api.cu: gb2)
  }
}

long long* g_tt_trace = nullptr;  // debug buffer [6 launches][4 layers][16] (brl_tt_trace)
// per-device state (function attributes and the time-out word live in a device's context: one process may drive several GPUs)
constexpr int TT_MAX_DEV = 64;
int* g_tt_status[TT_MAX_DEV] = {};
int tt_device() {
  int d = 0;
  cudaGetDevice(&d);
  return d < 0 || d >= TT_MAX_DEV ? 0 : d;
}
int* tt_status_word() {
  const int d = tt_device();
  if (!g_tt_status[d]) {
    cudaMalloc(&g_tt_status[d], sizeof(int));
    cudaMemset(g_tt_status[d], 0, sizeof(int));
  }
  return g_tt_status[d];
}
inline size_t al256(size_t v) { return (v + 255) & ~(size_t)255; }

#include "brl_tc_train_linear.cuh"
#include "brl_tc_train_convd3.cuh"

}  // namespace

void tt_trace(long long* device_buf) { g_tt_trace = device_buf; }

int tt_status() {  // of the current device
  int v = 0;
  const int d = tt_device();
  if (g_tt_status[d]) cudaMemcpy(&v, g_tt_status[d], sizeof(int), cudaMemcpyDeviceToHost);
  return v;
}

size_t tt_lane_bytes(long long B) {
  const size_t nt = (size_t)((B + 3) / 4);
  return al256(nt * 6 * CS) + al256(nt * 16 * CS) + 2 * al256(nt * 8 * CS) + 4 * al256(nt * 16 * CS) + 2 * al256(nt * 8 * CS) +
         al256(nt * RBUF_PER_TILE * sizeof(float)) + al256((size_t)table().blob_bytes) + al256(nt * (size_t)table().part_floats * sizeof(float)) +
         5 * al256((size_t)((B + 127) / 128) * FC_MT_BYTES) + al256(4 * (size_t)FC_WIMG) + 256;
}
void tt_carve(unsigned char* base, long long B, TtLane& ln) {
  const size_t nt = (size_t)((B + 3) / 4);
  unsigned char* p = reinterpret_cast<unsigned char*>(al256(reinterpret_cast<size_t>(base)));
  auto take = [&](size_t bytes) { unsigned char* r = p; p += al256(bytes); return r; };
  ln.ximg = take(nt * 6 * CS);
  ln.m1 = take(nt * 16 * CS);
  ln.t2 = take(nt * 8 * CS);
  ln.t3 = take(nt * 8 * CS);
  for (int k = 0; k < 4; ++k) ln.g[k] = take(nt * 16 * CS);
  ln.g[4] = take(nt * 8 * CS);
  ln.g[5] = take(nt * 8 * CS);
  ln.rbuf = reinterpret_cast<float*>(take(nt * RBUF_PER_TILE * sizeof(float)));
  ln.blob = take((size_t)table().blob_bytes);
  ln.part = reinterpret_cast<float*>(take(nt * (size_t)table().part_floats * sizeof(float)));  // at most one group per tile
  const size_t nmt = (size_t)((B + 127) / 128);
  ln.fimg = take(nmt * FC_MT_BYTES);
  ln.fbimg = take(nmt * FC_MT_BYTES);
  ln.f2img = take(nmt * FC_MT_BYTES);
  ln.f2bimg = take(nmt * FC_MT_BYTES);
  ln.gfimg = take(nmt * FC_MT_BYTES);
  ln.fcblob = take(4 * (size_t)FC_WIMG);
}

static void tt_configure() {
  static bool done_dev[TT_MAX_DEV] = {};
  bool& done = done_dev[tt_device()];
  if (done) return;
  cudaFuncSetAttribute(tt_fwd_kernel<BRL_MODE_LRT>, cudaFuncAttributeMaxDynamicSharedMemorySize, F_SMEM);
  cudaFuncSetAttribute(tt_fwd_kernel<BRL_MODE_FLIPOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, F_SMEM);
  cudaFuncSetAttribute(tt_fwd_kernel<TT_PLAIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, F_SMEM);
  cudaFuncSetAttribute(tt_bwd_kernel<TT_PLAIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, B_SMEM);
  cudaFuncSetAttribute(tt_fc_dx_kernel<TT_PLAIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, FX_SMEM);
  cudaFuncSetAttribute(tt_fc_dw_kernel<TT_PLAIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, FW_SMEM);
  cudaFuncSetAttribute(tt_bwd_kernel<BRL_MODE_LRT>, cudaFuncAttributeMaxDynamicSharedMemorySize, B_SMEM);
  cudaFuncSetAttribute(tt_bwd_kernel<BRL_MODE_FLIPOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, B_SMEM);
  cudaFuncSetAttribute(tt_fc_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, FF_SMEM);
  cudaFuncSetAttribute(tt_fc_dx_kernel<BRL_MODE_LRT>, cudaFuncAttributeMaxDynamicSharedMemorySize, FX_SMEM);
  cudaFuncSetAttribute(tt_fc_dx_kernel<BRL_MODE_FLIPOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, FX_SMEM);
  cudaFuncSetAttribute(tt_fc_dw_kernel<BRL_MODE_LRT>, cudaFuncAttributeMaxDynamicSharedMemorySize, FW_SMEM);
  cudaFuncSetAttribute(tt_fc_dw_kernel<BRL_MODE_FLIPOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, FW_SMEM);
  done = true;
}
static TtLayer layer_of(const TtStep& s, int i) {
  TtLayer l = table().L[i];
  l.w_off = s.w_off[i];
  l.b_off = s.b_off[i];
  return l;
}

void tt_forward(const TtLane& ln, const TtStep& s, cudaStream_t st, const TtSide& sd) {
  tt_configure();
  const int nt = (int)((s.B + 3) / 4);
  const Table& tb = table();
  cudaEventRecord(sd.fork, st);  // the parameters (and a Flipout weight draw) are complete on `st` here
  cudaStreamWaitEvent(sd.side, sd.fork, 0);
  const unsigned M = (unsigned)s.members;
  tt_packx_kernel<<<dim3((unsigned)(((long long)nt * 3 * ROWS + 255) / 256), 1, M), 256, 0, st>>>(s.x, ln.ximg, (int)s.B, nt, s.lane_stride);
  TtPackArgs pa;
  for (int i = 0; i < TT_LAYERS; ++i) { pa.L[i] = layer_of(s, i); pa.start[i] = tb.pack_start[i]; }
  pa.start[TT_LAYERS] = tb.pack_start[TT_LAYERS];
  pa.mode = s.mode; pa.mu = s.mu; pa.second = s.mode == BRL_MODE_LRT ? s.sigma : s.mode == BRL_MODE_FLIPOUT ? s.wsamp : s.mu; pa.blob = ln.blob;
  pa.P = s.P; pa.lane_stride = s.lane_stride;
  tt_pack_kernel<<<dim3((tb.pack_start[TT_LAYERS] + TT_LAYERS * 64 + 255) / 256, 1, M), 256, 0, sd.side>>>(pa);
  TtFcPackArgs fp;
  fp.mode = s.mode; fp.mu = s.mu; fp.second = pa.second; fp.w_off = s.w_off_fc; fp.blob = ln.fcblob;
  fp.P = s.P; fp.lane_stride = s.lane_stride;
  tt_pack_fc_kernel<<<dim3((64 * 2400 + 255) / 256, 1, M), 256, 0, sd.side>>>(fp);
  cudaEventRecord(sd.join, sd.side);
  g_launch_count += 3;
  if (s.B % 128 != 0) {  // windows beyond B of the last 128-window M-tile are K rows of the fc weight-gradient GEMM: they must be zero
    const size_t last = (size_t)(s.B / 128) * FC_MT_BYTES, pitch = M > 1 ? (size_t)s.lane_stride : FC_MT_BYTES;  // every member's
    cudaMemset2DAsync(ln.fbimg + last, pitch, 0, FC_MT_BYTES, M, st);
    cudaMemset2DAsync(ln.f2img + last, pitch, 0, FC_MT_BYTES, M, st);
    cudaMemset2DAsync(ln.f2bimg + last, pitch, 0, FC_MT_BYTES, M, st);
    cudaMemset2DAsync(ln.fimg + last, pitch, 0, FC_MT_BYTES, M, st);
  }
  cudaStreamWaitEvent(st, sd.join, 0);  // weight images ready
  static const int levels[3][4] = {{0, 1, 2, 3}, {5, 7, 4, 9}, {6, 8, -1, -1}};
  for (int lv = 0; lv < 3; ++lv) {
    TtFwdArgs fa{};
    fa.ln = ln;
    if (s.mode != BRL_MODE_LRT) fa.ln.rbuf = nullptr;
    fa.B = (int)s.B; fa.ntile = nt; fa.sgn_fc_in = s.sgn_fc_in; fa.lane_stride = s.lane_stride; fa.status = tt_status_word();
    fa.noise_stride = s.noise_stride; fa.sign_stride = s.sign_stride;
    fa.trace = g_tt_trace ? g_tt_trace + lv * 64 : nullptr;
    int nl = 0;
    for (int k = 0; k < 4; ++k) {
      const int li = levels[lv][k];
      if (li < 0) continue;
      fa.lay[nl] = layer_of(s, li);
      fa.eps[nl] = s.eps[li];
      fa.sgn_in[nl] = s.sgn_in[li];
      fa.sgn_out[nl] = s.sgn_out[li];
      fa.drop[nl] = s.drop[li];
      fa.keep[nl] = s.keep[li];
      ++nl;
    }
    fa.nl = nl;
    ++g_launch_count;
    if (s.mode == BRL_MODE_LRT) tt_fwd_kernel<BRL_MODE_LRT><<<dim3(nt, nl, M), NT, F_SMEM, st>>>(fa);
    else if (s.mode == BRL_MODE_FLIPOUT) tt_fwd_kernel<BRL_MODE_FLIPOUT><<<dim3(nt, nl, M), NT, F_SMEM, st>>>(fa);
    else tt_fwd_kernel<TT_PLAIN><<<dim3(nt, nl, M), NT, F_SMEM, st>>>(fa);
  }
}

void tt_fc_forward(const TtLane& ln, const TtStep& s, float* part, cudaStream_t st) {
  tt_configure();
  const int nmt = (int)((s.B + 127) / 128);
  cudaMemsetAsync(part, 0, sizeof(float) * 2 * (size_t)s.B * 64 * s.members, st);  // [members][2][B][64]
  TtFcFwdArgs fa{};
  fa.ln = ln; fa.B = (int)s.B; fa.mode = s.mode; fa.part = part; fa.status = tt_status_word();
  fa.lane_stride = s.lane_stride; fa.part_stride = 2 * s.B * 64;
  ++g_launch_count;
  tt_fc_fwd_kernel<<<dim3(nmt, FC_KS, s.members), 256, FF_SMEM, st>>>(fa);
}

void tt_tail(const TtStep& s, const TtTail& t, cudaStream_t st) {
  TtTailArgs a{};
  a.B = (int)s.B; a.mode = s.mode; a.compute_grads = t.compute_grads;
  a.part = t.part;
  const bool lrt = s.mode == BRL_MODE_LRT, plain = s.mode != BRL_MODE_LRT && s.mode != BRL_MODE_FLIPOUT;
  a.fc_b0 = ((lrt || plain) ? s.mu : s.wsamp) + s.b_off_fc; a.fc_b1 = lrt ? s.sigma + s.b_off_fc : nullptr;
  a.hw0 = s.mu + t.hw_off; a.hw1 = plain ? nullptr : (lrt ? s.sigma : s.wsamp) + t.hw_off;
  a.hb0 = ((lrt || plain) ? s.mu : s.wsamp) + t.hb_off; a.hb1 = lrt ? s.sigma + t.hb_off : nullptr;
  a.loss_kind = t.loss_kind; a.keep_fc = t.keep_fc; a.drop_fc = t.drop_fc;
  a.eps_fc = t.eps_fc; a.eps_head = t.eps_head;
  a.sout_fc = t.sout_fc; a.sin_head = t.sin_head; a.sout_head = t.sout_head;
  a.y = t.y; a.gscale = t.gscale; a.acc = t.acc; a.out = t.out; a.dpre = t.dpre; a.dsec = t.dsec;
  a.g0 = s.g0; a.g1 = s.g1; a.hw_off = t.hw_off; a.hb_off = t.hb_off;
  a.P = s.P; a.part_stride = 2 * s.B * t.width;
  a.noise_stride = s.noise_stride; a.sign_stride = s.sign_stride; a.acc_stride = t.acc_stride;
  const dim3 grid((unsigned)std::min<long long>((s.B + 7) / 8, 148), 1, (unsigned)s.members);
  ++g_launch_count;
  if (t.width == 320) {
    if (lrt) tt_tail_kernel<BRL_MODE_LRT, 320><<<grid, 256, 0, st>>>(a);
    else if (plain) tt_tail_kernel<TT_PLAIN, 320><<<grid, 256, 0, st>>>(a);
    else tt_tail_kernel<BRL_MODE_FLIPOUT, 320><<<grid, 256, 0, st>>>(a);
  } else if (t.width == 32) {
    if (lrt) tt_tail_kernel<BRL_MODE_LRT, 32><<<grid, 256, 0, st>>>(a);
    else if (plain) tt_tail_kernel<TT_PLAIN, 32><<<grid, 256, 0, st>>>(a);
    else tt_tail_kernel<BRL_MODE_FLIPOUT, 32><<<grid, 256, 0, st>>>(a);
  } else {
    if (lrt) tt_tail_kernel<BRL_MODE_LRT, 64><<<grid, 256, 0, st>>>(a);
    else if (plain) tt_tail_kernel<TT_PLAIN, 64><<<grid, 256, 0, st>>>(a);
    else tt_tail_kernel<BRL_MODE_FLIPOUT, 64><<<grid, 256, 0, st>>>(a);
  }
}

void tt_fc_backward(const TtLane& ln, const TtStep& s, const float* dpre, const float* dsec, cudaStream_t st, const TtSide& sd) {
  tt_configure();
  TtFcBwdArgs ba{};
  ba.ln = ln; ba.B = (int)s.B; ba.nmt = (int)((s.B + 127) / 128); ba.mode = s.mode; ba.dpre = dpre; ba.dsec = dsec;
  ba.sgn_in = s.sgn_fc_in; ba.g0 = s.g0; ba.g1 = s.g1; ba.w_off = s.w_off_fc; ba.b_off = s.b_off_fc; ba.status = tt_status_word();
  ba.P = s.P; ba.lane_stride = s.lane_stride;
  g_launch_count += 2;
  // the weight gradient needs nothing downstream of it until the finalisation: it leaves the critical chain for the side stream
  // (joined at the end of tt_backward)
  cudaEventRecord(sd.fork, st);
  cudaStreamWaitEvent(sd.side, sd.fork, 0);
  if (s.mode == BRL_MODE_LRT) {
    tt_fc_dx_kernel<BRL_MODE_LRT><<<dim3(ba.nmt, FC_NS, s.members), 256, FX_SMEM, st>>>(ba);
    tt_fc_dw_kernel<BRL_MODE_LRT><<<dim3((FC_KC + 15) / 16, 1, s.members), 256, FW_SMEM, sd.side>>>(ba);
  } else if (s.mode != BRL_MODE_FLIPOUT) {
    tt_fc_dx_kernel<TT_PLAIN><<<dim3(ba.nmt, FC_NS, s.members), 256, FX_SMEM, st>>>(ba);
    tt_fc_dw_kernel<TT_PLAIN><<<dim3((FC_KC + 15) / 16, 1, s.members), 256, FW_SMEM, sd.side>>>(ba);
  } else {
    tt_fc_dx_kernel<BRL_MODE_FLIPOUT><<<dim3(ba.nmt, FC_NS, s.members), 256, FX_SMEM, st>>>(ba);
    tt_fc_dw_kernel<BRL_MODE_FLIPOUT><<<dim3((FC_KC + 15) / 16, 1, s.members), 256, FW_SMEM, sd.side>>>(ba);
  }
  cudaEventRecord(sd.join, sd.side);
}

void tt_backward(const TtLane& ln, const TtStep& s, cudaStream_t st, const TtSide& sd) {
  tt_configure();
  const int nt = (int)((s.B + 3) / 4);
  // reverse dependency levels: {b2b, b3b, b1, b4} need only the fc layer's gradient; {b2a, b3a} need d/dT2, d/dT3;
  // module 1 needs the four d/dM1 images
  static const int levels[3][4] = {{6, 8, 4, 9}, {5, 7, -1, -1}, {2, 1, 3, 0}};
  const Table& tb = table();
  TtReduceArgs ra{};
  for (int lv = 0; lv < 3; ++lv) {
    TtBwdArgs ba{};
    ba.ln = ln;
    ba.part_floats = tb.part_floats;
    ba.B = (int)s.B; ba.ntile = nt; ba.g0 = s.g0; ba.g1 = s.g1; ba.lane_stride = s.lane_stride; ba.status = tt_status_word();
    ba.sign_stride = s.sign_stride;
    ba.trace = g_tt_trace ? g_tt_trace + (3 + lv) * 64 : nullptr;
    int nl = 0;
    for (int k = 0; k < 4; ++k) {
      const int li = levels[lv][k];
      if (li < 0) continue;
      ba.lay[nl] = layer_of(s, li);
      ba.sgn_in[nl] = s.sgn_in[li];
      ba.sgn_out[nl] = s.sgn_out[li];
      ba.keep[nl] = s.keep[li];
      ++nl;
    }
    ba.nl = nl;
    ba.tiles_per_cta = std::max(1, (nt * nl * s.members + 147) / 148);  // about one wave of 148 CTAs over all members
    const int ngroups = (nt + ba.tiles_per_cta - 1) / ba.tiles_per_cta;
    for (int k = 0; k < 4; ++k)
      if (levels[lv][k] >= 0) ra.ngroups[levels[lv][k]] = ngroups;
    ++g_launch_count;
    const dim3 grid(ngroups, nl, s.members);
    if (s.mode == BRL_MODE_LRT) tt_bwd_kernel<BRL_MODE_LRT><<<grid, NT, B_SMEM, st>>>(ba);
    else if (s.mode == BRL_MODE_FLIPOUT) tt_bwd_kernel<BRL_MODE_FLIPOUT><<<grid, NT, B_SMEM, st>>>(ba);
    else tt_bwd_kernel<TT_PLAIN><<<grid, NT, B_SMEM, st>>>(ba);
  }
  int tot = 0;
  for (int i = 0; i < TT_LAYERS; ++i) {
    ra.L[i] = layer_of(s, i);
    ra.start[i] = tot;
    tot += ra.L[i].N * ra.L[i].T * ra.L[i].KC * 8 + ra.L[i].N;
  }
  ra.start[TT_LAYERS] = tot;
  ra.part_floats = tb.part_floats; ra.mode = s.mode; ra.part = ln.part; ra.g0 = s.g0; ra.g1 = s.g1;
  ra.P = s.P; ra.lane_stride = s.lane_stride;
  ++g_launch_count;
  tt_reduce_kernel<<<dim3((tot + 255) / 256, RED_SPLIT, s.members), 256, 0, st>>>(ra);
  cudaStreamWaitEvent(st, sd.join, 0);  // the fc weight gradient (tt_fc_backward) is part of what the caller finalises next
}

// ---- Linear net (brl_tc_train_linear.cuh) --------------------------------------------------------------------------------
size_t tl_lane_bytes(long long B) {
  const size_t nmt = (size_t)((B + 127) / 128);
  size_t b = 256;
  for (int l = 0; l < 4; ++l) b += 4 * al256(nmt * tl_kc(l) * TL_CH) + al256(4 * (size_t)tl_wimg(l));
  for (int l = 0; l < 3; ++l) b += al256((size_t)B * tl_n(l) * sizeof(float));
  return b + al256(2 * (size_t)B * 32 * sizeof(float));
}
void tl_carve(unsigned char* base, long long B, TlLane& ln) {
  const size_t nmt = (size_t)((B + 127) / 128);
  unsigned char* p = reinterpret_cast<unsigned char*>(al256(reinterpret_cast<size_t>(base)));
  auto take = [&](size_t bytes) { unsigned char* r = p; p += al256(bytes); return r; };
  for (int l = 0; l < 4; ++l) {
    for (int k = 0; k < 4; ++k) ln.act[l][k] = take(nmt * tl_kc(l) * TL_CH);
    ln.w[l] = take(4 * (size_t)tl_wimg(l));
  }
  for (int l = 0; l < 3; ++l) ln.rbuf[l] = reinterpret_cast<float*>(take((size_t)B * tl_n(l) * sizeof(float)));
  ln.part = reinterpret_cast<float*>(take(2 * (size_t)B * 32 * sizeof(float)));
}

static void tl_configure() {
  static bool done_dev[TT_MAX_DEV] = {};
  bool& done = done_dev[tt_device()];
  if (done) return;
  cudaFuncSetAttribute(tl_fwd_kernel<BRL_MODE_LRT>, cudaFuncAttributeMaxDynamicSharedMemorySize, TLF_SMEM);
  cudaFuncSetAttribute(tl_fwd_kernel<BRL_MODE_FLIPOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, TLF_SMEM);
  cudaFuncSetAttribute(tl_fwd_kernel<TT_PLAIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, TLF_SMEM);
  cudaFuncSetAttribute(tl_dx_kernel<BRL_MODE_LRT>, cudaFuncAttributeMaxDynamicSharedMemorySize, TLX_SMEM);
  cudaFuncSetAttribute(tl_dx_kernel<BRL_MODE_FLIPOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, TLX_SMEM);
  cudaFuncSetAttribute(tl_dx_kernel<TT_PLAIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, TLX_SMEM);
  cudaFuncSetAttribute(tl_dw_kernel<BRL_MODE_LRT>, cudaFuncAttributeMaxDynamicSharedMemorySize, TLW_SMEM);
  cudaFuncSetAttribute(tl_dw_kernel<BRL_MODE_FLIPOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, TLW_SMEM);
  cudaFuncSetAttribute(tl_dw_kernel<TT_PLAIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, TLW_SMEM);
  done = true;
}

void tl_forward(const TlLane& ln, const TtStep& s, cudaStream_t st, const TtSide& sd) {
  tl_configure();
  const int B = (int)s.B, nmt = (B + 127) / 128;
  const bool lrt = s.mode == BRL_MODE_LRT, flip = s.mode == BRL_MODE_FLIPOUT;
  cudaEventRecord(sd.fork, st);  // the parameters (and a weight draw) are complete on `st` here
  cudaStreamWaitEvent(sd.side, sd.fork, 0);
  TlPackWArgs pw{};
  pw.mode = s.mode; pw.mu = s.mu; pw.second = lrt ? s.sigma : flip ? s.wsamp : s.mu;
  for (int l = 0; l < 4; ++l) { pw.w_off[l] = s.w_off[l]; pw.w[l] = ln.w[l]; }
  tl_pack_w_kernel<<<(TL_PACK_END + 255) / 256, 256, 0, sd.side>>>(pw);
  cudaEventRecord(sd.join, sd.side);
  TlPackXArgs px{};
  px.x = s.x; px.sgn_in = s.sgn_in[0]; px.B = B; px.mode = s.mode;
  for (int k = 0; k < 4; ++k) px.img[k] = ln.act[0][k];
  tl_packx_kernel<<<(unsigned)(((long long)nmt * 72 * 128 + 255) / 256), 256, 0, st>>>(px);
  cudaStreamWaitEvent(st, sd.join, 0);  // weight images ready
  g_launch_count += 6;
  for (int l = 0; l < 4; ++l) {
    TlFwdArgs fa{};
    fa.a0 = ln.act[l][0]; fa.a1 = ln.act[l][2];
    fa.w0 = ln.w[l]; fa.w1 = ln.w[l] + (flip ? 3 : 2) * (size_t)tl_wimg(l);
    fa.B = B; fa.N = tl_n(l); fa.KC = tl_kc(l); fa.last = l == 3;
    fa.b0 = (flip ? s.wsamp : s.mu) + s.b_off[l]; fa.b1 = lrt ? s.sigma + s.b_off[l] : nullptr;
    fa.eps = s.eps[l]; fa.drop = s.drop[l]; fa.keep = s.keep[l];
    fa.sout = s.sgn_out[l]; fa.sin_next = s.sgn_in[l + 1];
    if (l < 3)
      for (int k = 0; k < 4; ++k) fa.out[k] = ln.act[l + 1][k];
    fa.rbuf = l < 3 ? ln.rbuf[l] : nullptr; fa.part = ln.part; fa.status = tt_status_word();
    const dim3 grid(nmt, tl_n(l) / TL_NS);
    if (lrt) tl_fwd_kernel<BRL_MODE_LRT><<<grid, 128, TLF_SMEM, st>>>(fa);
    else if (flip) tl_fwd_kernel<BRL_MODE_FLIPOUT><<<grid, 128, TLF_SMEM, st>>>(fa);
    else tl_fwd_kernel<TT_PLAIN><<<grid, 128, TLF_SMEM, st>>>(fa);
  }
}

void tl_backward(const TlLane& ln, const TtStep& s, float* const* dpre, float* const* dsec, cudaStream_t st, const TtSide& sd) {
  tl_configure();
  const int B = (int)s.B, nmt = (B + 127) / 128;
  const bool lrt = s.mode == BRL_MODE_LRT, flip = s.mode == BRL_MODE_FLIPOUT;
  for (int l = 3; l >= 0; --l) {
    // weight gradient of layer l: needs nothing downstream of it until the finalisation, so it runs on the side stream
    cudaEventRecord(sd.fork, st);
    cudaStreamWaitEvent(sd.side, sd.fork, 0);
    TlDwArgs wa{};
    wa.a0 = ln.act[l][1]; wa.a1 = ln.act[l][lrt ? 2 : 3]; wa.g0 = dpre[l]; wa.g1 = dsec[l];
    wa.B = B; wa.N = tl_n(l); wa.KC = tl_kc(l); wa.cin = tl_cin(l); wa.nsl = std::min(TL_WS, tl_n(l)); wa.mt_per = nmt;
    wa.gw0 = s.g0; wa.gw1 = s.g1; wa.w_off = s.w_off[l]; wa.b_off = s.b_off[l]; wa.status = tt_status_word();
    const dim3 wgrid((tl_kc(l) + 15) / 16, tl_n(l) / wa.nsl);
    if (lrt) tl_dw_kernel<BRL_MODE_LRT><<<wgrid, 256, TLW_SMEM, sd.side>>>(wa);
    else if (flip) tl_dw_kernel<BRL_MODE_FLIPOUT><<<wgrid, 256, TLW_SMEM, sd.side>>>(wa);
    else tl_dw_kernel<TT_PLAIN><<<wgrid, 256, TLW_SMEM, sd.side>>>(wa);
    ++g_launch_count;
    if (l == 0) break;  // layer 0's input is x: no input gradient
    TlDxArgs xa{};
    xa.g0 = dpre[l]; xa.g1 = dsec[l];
    xa.w0 = ln.w[l] + tl_wimg(l); xa.w1 = ln.w[l] + 2 * (size_t)tl_wimg(l); xa.act = ln.act[l][0];
    xa.B = B; xa.Nl = tl_n(l); xa.KCl = tl_kc(l);
    xa.sin_ = s.sgn_in[l]; xa.rb = ln.rbuf[l - 1]; xa.sout = s.sgn_out[l - 1]; xa.keep = s.keep[l - 1];
    xa.d0 = dpre[l - 1]; xa.d1 = dsec[l - 1]; xa.status = tt_status_word();
    const dim3 xgrid(nmt, tl_cin(l) / TL_XS);
    if (lrt) tl_dx_kernel<BRL_MODE_LRT><<<xgrid, 256, TLX_SMEM, st>>>(xa);
    else if (flip) tl_dx_kernel<BRL_MODE_FLIPOUT><<<xgrid, 256, TLX_SMEM, st>>>(xa);
    else tl_dx_kernel<TT_PLAIN><<<xgrid, 256, TLX_SMEM, st>>>(xa);
    ++g_launch_count;
  }
  cudaEventRecord(sd.join, sd.side);
  cudaStreamWaitEvent(st, sd.join, 0);  // the weight gradients are part of what the caller finalises next
}

// ---- Conv-D3 net (brl_tc_train_convd3.cuh) -------------------------------------------------------------------------------
size_t tc3_lane_bytes(long long B) {
  size_t b = 256;
  for (int l = 0; l < 3; ++l) {
    const size_t M = (size_t)B * tc3_p(l), nmt = (M + 127) / 128;
    b += 4 * al256(nmt * tc3_kc(l) * TL_CH) + al256(4 * (size_t)tc3_wimg(l)) + 4 * al256(M * tc3_n(l) * sizeof(float));
  }
  return b + 2 * al256((size_t)B * 25 * 320 * sizeof(float)) + 2 * al256((size_t)B * 320 * sizeof(float));
}
void tc3_carve(unsigned char* base, long long B, Tc3Lane& ln) {
  unsigned char* p = reinterpret_cast<unsigned char*>(al256(reinterpret_cast<size_t>(base)));
  auto take = [&](size_t bytes) { unsigned char* r = p; p += al256(bytes); return r; };
  auto takef = [&](size_t n) { return reinterpret_cast<float*>(take(n * sizeof(float))); };
  for (int l = 0; l < 3; ++l) {
    const size_t M = (size_t)B * tc3_p(l), nmt = (M + 127) / 128;
    for (int k = 0; k < 4; ++k) ln.img[l][k] = take(nmt * tc3_kc(l) * TL_CH);
    ln.w[l] = take(4 * (size_t)tc3_wimg(l));
    ln.act[l] = takef(M * tc3_n(l));
    ln.rbuf[l] = takef(M * tc3_n(l));
    ln.g[l][0] = takef(M * tc3_n(l));
    ln.g[l][1] = takef(M * tc3_n(l));
  }
  ln.col[0] = takef((size_t)B * 25 * 320);
  ln.col[1] = takef((size_t)B * 25 * 320);
  ln.feat = takef((size_t)B * 320);
  ln.dfeat = takef((size_t)B * 320);
}

static void tc3_configure() {
  static bool done_dev[TT_MAX_DEV] = {};
  bool& done = done_dev[tt_device()];
  if (done) return;
  tl_configure();  // tl_dx_kernel / tl_dw_kernel
  cudaFuncSetAttribute(tc3_fwd_kernel<BRL_MODE_LRT>, cudaFuncAttributeMaxDynamicSharedMemorySize, TLF_SMEM);
  cudaFuncSetAttribute(tc3_fwd_kernel<BRL_MODE_FLIPOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, TLF_SMEM);
  cudaFuncSetAttribute(tc3_fwd_kernel<TT_PLAIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, TLF_SMEM);
  done = true;
}

void tc3_forward(const Tc3Lane& ln, const TtStep& s, cudaStream_t st, const TtSide& sd) {
  tc3_configure();
  const int B = (int)s.B;
  const bool lrt = s.mode == BRL_MODE_LRT, flip = s.mode == BRL_MODE_FLIPOUT;
  cudaEventRecord(sd.fork, st);  // the parameters (and a weight draw) are complete on `st` here
  cudaStreamWaitEvent(sd.side, sd.fork, 0);
  Tc3PackWArgs pw{};
  pw.mode = s.mode; pw.mu = s.mu; pw.second = lrt ? s.sigma : flip ? s.wsamp : s.mu;
  for (int l = 0; l < 3; ++l) { pw.w_off[l] = s.w_off[l]; pw.w[l] = ln.w[l]; }
  tc3_pack_w_kernel<<<(TC3_PACK_END + 255) / 256, 256, 0, sd.side>>>(pw);
  cudaEventRecord(sd.join, sd.side);
  g_launch_count += 8;
  for (int l = 0; l < 3; ++l) {
    const int M = B * tc3_p(l), nmt = (M + 127) / 128;
    Tc3Im2colArgs ia{};
    ia.l = l; ia.B = B; ia.mode = s.mode; ia.src = l == 0 ? s.x : ln.act[l - 1]; ia.sgn_in = s.sgn_in[l];
    for (int k = 0; k < 4; ++k) ia.img[k] = ln.img[l][k];
    tc3_im2col_kernel<<<(unsigned)(((long long)nmt * tc3_kc(l) * 128 + 255) / 256), 256, 0, st>>>(ia);
    if (l == 0) cudaStreamWaitEvent(st, sd.join, 0);  // weight images ready
    Tc3FwdArgs fa{};
    fa.a0 = ln.img[l][0]; fa.a1 = ln.img[l][2];
    fa.w0 = ln.w[l]; fa.w1 = ln.w[l] + (flip ? 3 : 2) * (size_t)tc3_wimg(l);
    fa.B = B; fa.N = tc3_n(l); fa.P = tc3_p(l); fa.KC = tc3_kc(l);
    fa.b0 = (flip ? s.wsamp : s.mu) + s.b_off[l]; fa.b1 = lrt ? s.sigma + s.b_off[l] : nullptr;
    fa.eps = s.eps[l]; fa.drop = s.drop[l]; fa.keep = s.keep[l]; fa.sout = s.sgn_out[l];
    fa.act = ln.act[l]; fa.rbuf = ln.rbuf[l]; fa.status = tt_status_word();
    const dim3 grid(nmt, tc3_nimg(l) / TL_NS);
    if (lrt) tc3_fwd_kernel<BRL_MODE_LRT><<<grid, 128, TLF_SMEM, st>>>(fa);
    else if (flip) tc3_fwd_kernel<BRL_MODE_FLIPOUT><<<grid, 128, TLF_SMEM, st>>>(fa);
    else tc3_fwd_kernel<TT_PLAIN><<<grid, 128, TLF_SMEM, st>>>(fa);
  }
  tc3_pool_kernel<<<(B * 320 + 255) / 256, 256, 0, st>>>(ln.act[2], ln.feat, B);
}

void tc3_backward(const Tc3Lane& ln, const TtStep& s, cudaStream_t st, const TtSide& sd) {
  tc3_configure();
  const int B = (int)s.B;
  const bool lrt = s.mode == BRL_MODE_LRT, flip = s.mode == BRL_MODE_FLIPOUT;
  auto act_bwd = [&](int l, const float* src0, const float* src1) {
    Tc3ActBwdArgs aa{};
    aa.l = l; aa.B = B; aa.mode = lrt ? BRL_MODE_LRT : flip ? BRL_MODE_FLIPOUT : TT_PLAIN; aa.keep = s.keep[l];
    aa.src0 = src0; aa.src1 = src1; aa.act = ln.act[l]; aa.rb = ln.rbuf[l]; aa.sout = s.sgn_out[l]; aa.sin_next = s.sgn_in[l + 1];
    aa.d0 = ln.g[l][0]; aa.d1 = ln.g[l][1];
    const long long n = (long long)B * tc3_p(l) * tc3_n(l);
    tc3_bwd_act_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(aa);
    ++g_launch_count;
  };
  act_bwd(2, ln.dfeat, nullptr);
  for (int l = 2; l >= 0; --l) {
    const int M = B * tc3_p(l), nmt = (M + 127) / 128;
    // weight gradient of conv l: needs nothing downstream of it until the finalisation, so it runs on the side stream; its M-tiles
    // are split so that the launch covers the GPU (conv1: 520 M-tiles at B = 256)
    cudaEventRecord(sd.fork, st);
    cudaStreamWaitEvent(sd.side, sd.fork, 0);
    TlDwArgs wa{};
    wa.a0 = ln.img[l][1]; wa.a1 = ln.img[l][lrt ? 2 : 3]; wa.g0 = ln.g[l][0]; wa.g1 = ln.g[l][1];
    wa.B = M; wa.N = tc3_n(l); wa.KC = tc3_kc(l); wa.cin = tc3_k(l); wa.nsl = tc3_n(l);
    const int kt = (tc3_kc(l) + 15) / 16, split = std::max(1, std::min(nmt, 148 / kt));
    wa.mt_per = (nmt + split - 1) / split; wa.atomic = 1;
    wa.gw0 = s.g0; wa.gw1 = s.g1; wa.w_off = s.w_off[l]; wa.b_off = s.b_off[l]; wa.status = tt_status_word();
    const dim3 wgrid(kt, 1, (nmt + wa.mt_per - 1) / wa.mt_per);
    if (lrt) tl_dw_kernel<BRL_MODE_LRT><<<wgrid, 256, TLW_SMEM, sd.side>>>(wa);
    else if (flip) tl_dw_kernel<BRL_MODE_FLIPOUT><<<wgrid, 256, TLW_SMEM, sd.side>>>(wa);
    else tl_dw_kernel<TT_PLAIN><<<wgrid, 256, TLW_SMEM, sd.side>>>(wa);
    ++g_launch_count;
    if (l == 0) break;  // conv1's input is x: no input gradient
    TlDxArgs xa{};
    xa.g0 = ln.g[l][0]; xa.g1 = ln.g[l][1];
    xa.w0 = ln.w[l] + tc3_wimg(l); xa.w1 = ln.w[l] + 2 * (size_t)tc3_wimg(l);
    xa.B = M; xa.Nl = tc3_n(l); xa.KCl = tc3_kc(l); xa.keep = 1.0f; xa.raw = 1;
    xa.d0 = ln.col[0]; xa.d1 = ln.col[1]; xa.status = tt_status_word();
    const dim3 xgrid(nmt, tc3_kc(l) * 8 / TL_XS);
    if (lrt) tl_dx_kernel<BRL_MODE_LRT><<<xgrid, 256, TLX_SMEM, st>>>(xa);
    else if (flip) tl_dx_kernel<BRL_MODE_FLIPOUT><<<xgrid, 256, TLX_SMEM, st>>>(xa);
    else tl_dx_kernel<TT_PLAIN><<<xgrid, 256, TLX_SMEM, st>>>(xa);
    ++g_launch_count;
    act_bwd(l - 1, ln.col[0], ln.col[1]);
  }
  cudaEventRecord(sd.join, sd.side);
  cudaStreamWaitEvent(st, sd.join, 0);  // the weight gradients are part of what the caller finalises next
}

}  // namespace brl
