// Level-fused tcgen05 training kernels of the Conv-D3 net (conv.py:47-61,73-77: x.unsqueeze(1) [1,30,18] -> Conv2d(1,16,(5,9)) ->
// ReLU -> Conv2d(16,32,(2,10)) -> ReLU -> AvgPool((2,1)) -> Conv2d(32,64,(2,1)) -> ReLU -> AvgPool((2,1)) -> flatten 320 -> Linear(320,2),
// dropout sites behind the three convs).  Included by brl_tc_train.cu after the Linear net's file, whose kernels it reuses.
//
// Every conv is a dense GEMM whose rows are (window, output position), m = b * P + pos (P = 260, 25, 11), and whose K is the torch
// flatten order of the weight, k = (c * kh_n + kh) * kw_n + kw (K = 45 -> 64, 320, 64).  An im2col kernel writes a layer's input as
// operand images in the Linear net's chunk layout
//     [M-tile of 128 rows][K/8 chunks][128 rows][8 x 16 bit]      (rows beyond B * P are zero: they are K rows of the weight gradient)
// (the average pool in front of conv3 is applied while gathering), and the weight images are the Linear net's [N/32][K/8][32][8]
// (conv1's 16 outputs padded to 32).  So the three contractions are those of brl_tc_train_linear.cuh, on the same kernels:
//     forward           tl_fwd_mainloop + tc3_fwd_kernel's epilogue (bias, eps * sd / sign flips, ReLU, dropout; keyed by (b, n, pos)
//                       exactly as the fp32 back-end's gemm_epilogue, so native noise draws the same numbers)
//     input gradient    tl_dx_kernel with `raw` = 1: the [M, K] column gradients of conv3 / conv2, which tc3_bwd_act_kernel folds back
//                       (col2im), combines with the second path, routes through the pool and gates with the stored activation
//     weight gradient   tl_dw_kernel with its M-tiles split over gridDim.z CTAs and atomics (conv1 has 260 rows per window)
// The head stays in tt_tail_kernel (width 320, features as given).  Activations travel between launches as compact fp32 [M, N].
// Launches of one particle: weight packing (side stream) + 3 x (im2col, forward) + pool, the tail, then activation backward of conv3,
// 2 x (input gradient, col2im / activation backward) on the critical chain and three weight gradients on the side stream.

__host__ __device__ constexpr int tc3_n(int l) { return l == 0 ? 16 : l == 1 ? 32 : 64; }     // output channels
__host__ __device__ constexpr int tc3_p(int l) { return l == 0 ? 260 : l == 1 ? 25 : 11; }    // output positions per window
__host__ __device__ constexpr int tc3_k(int l) { return l == 0 ? 45 : l == 1 ? 320 : 64; }    // real K = Cin * kh * kw
__host__ __device__ constexpr int tc3_kc(int l) { return l == 1 ? 40 : 8; }                   // chunks of K (padded to 64 features)
__host__ __device__ constexpr int tc3_nimg(int l) { return l == 2 ? 64 : 32; }                // weight image rows (N padded to 32)
__host__ __device__ constexpr int tc3_wimg(int l) { return tc3_nimg(l) * tc3_kc(l) * 16; }    // bytes of one weight image
constexpr int TC3_PACK_END = 32 * 64 + 32 * 320 + 64 * 64;  // weight image elements of the three convs

struct Tc3PackWArgs {
  int mode;
  const float *mu, *second;  // second: sigma (LRT) or the weight draw (Flipout)
  long long w_off[3];
  unsigned char* w[3];       // fp16 mu | bf16 mu | bf16 sigma^2 or (W - mu) | fp16 (W - mu)
};
__global__ void tc3_pack_w_kernel(const Tc3PackWArgs a) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= TC3_PACK_END) return;
  int l = 0;
  while (j >= tc3_nimg(l) * tc3_kc(l) * 8) { j -= tc3_nimg(l) * tc3_kc(l) * 8; ++l; }
  const int K8 = tc3_kc(l) * 8, K = tc3_k(l), n = j / K8, k = j - n * K8;
  float m = 0.f, s = 0.f;
  const long long w_off = l == 0 ? a.w_off[0] : l == 1 ? a.w_off[1] : a.w_off[2];
  unsigned char* w = l == 0 ? a.w[0] : l == 1 ? a.w[1] : a.w[2];
  if (k < K && n < tc3_n(l)) {
    const long long wi = w_off + (long long)n * K + k;
    m = a.mu[wi];
    const float v = a.second[wi];
    s = a.mode == BRL_MODE_LRT ? v * v : a.mode == BRL_MODE_FLIPOUT ? v - m : 0.f;
  }
  const int o = (((n >> 5) * tc3_kc(l) + (k >> 3)) * 32 + (n & 31)) * 16 + (k & 7) * 2, img = tc3_wimg(l);
  *reinterpret_cast<__half*>(w + o) = __float2half_rn(m);
  *reinterpret_cast<__nv_bfloat16*>(w + img + o) = __float2bfloat16_rn(m);
  *reinterpret_cast<__nv_bfloat16*>(w + 2 * img + o) = __float2bfloat16_rn(s);
  *reinterpret_cast<__half*>(w + 3 * img + o) = __float2half_rn(s);
}

// im2col of conv l's input into its four operand images (same roles as tl_packx_kernel): thread = 8 features of one row
struct Tc3Im2colArgs {
  int l, B, mode;
  const float* src;     // l = 0: x [B, 30, 18]; else the previous conv's activation [B * P, N]
  const float* sgn_in;  // Flipout: s_in of conv l [B, Cin]
  unsigned char* img[4];
};
__global__ void tc3_im2col_kernel(const Tc3Im2colArgs a) {
  const int l = a.l, KC = tc3_kc(l), P = tc3_p(l), M = a.B * P;
  const long long u = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const int nmt = (M + 127) >> 7;
  if (u >= (long long)nmt * KC * 128) return;
  const int r = (int)(u & 127), c = (int)((u >> 7) % KC), mt = (int)((u >> 7) / KC), m = mt * 128 + r;
  const int b = m / P, pos = m - b * P;
  float f[8], s[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int k = c * 8 + j;
    float v = 0.f, sg = 1.f;
    if (m < M && k < tc3_k(l)) {
      if (l == 0) {  // k = kh * 9 + kw; pos = oh * 10 + ow
        const int kh = k / 9, kw = k - kh * 9, oh = pos / 10, ow = pos - oh * 10;
        v = a.src[(long long)b * 540 + (oh + kh) * 18 + ow + kw];
        if (a.mode == BRL_MODE_FLIPOUT) sg = a.sgn_in[b];
      } else if (l == 1) {  // k = (ci * 2 + kh) * 10 + kw over conv1's output [26 x 10]
        const int ci = k / 20, kh = (k / 10) & 1, kw = k % 10;
        v = a.src[((long long)b * 260 + (pos + kh) * 10 + kw) * 16 + ci];
        if (a.mode == BRL_MODE_FLIPOUT) sg = a.sgn_in[b * 16 + ci];
      } else {  // k = ci * 2 + kh over AvgPool((2,1)) of conv2's output: row t = pos + kh averages rows 2t, 2t + 1
        const int ci = k >> 1, t = pos + (k & 1);
        const float* p = a.src + ((long long)b * 25 + 2 * t) * 32 + ci;
        v = 0.5f * (p[0] + p[32]);
        if (a.mode == BRL_MODE_FLIPOUT) sg = a.sgn_in[b * 32 + ci];
      }
    }
    f[j] = __half2float(__float2half_rn(v));
    s[j] = a.mode == BRL_MODE_LRT ? f[j] * f[j] : a.mode == BRL_MODE_FLIPOUT ? f[j] * sg : 0.f;
  }
  const long long o = (long long)u * 16;
  *reinterpret_cast<uint4*>(a.img[0] + o) = pack_h8(f);
  *reinterpret_cast<uint4*>(a.img[1] + o) = pack_b8(f);
  if (a.mode == BRL_MODE_LRT) {
    *reinterpret_cast<uint4*>(a.img[2] + o) = pack_b8(s);
  } else if (a.mode == BRL_MODE_FLIPOUT) {
    *reinterpret_cast<uint4*>(a.img[2] + o) = pack_h8(s);
    *reinterpret_cast<uint4*>(a.img[3] + o) = pack_b8(s);
  }
}

// forward of conv l: one CTA = one 128-row M-tile x one 32-column weight slice (tl_fwd_mainloop); thread = row
struct Tc3FwdArgs {
  const unsigned char *a0, *a1, *w0, *w1;  // as TlFwdArgs
  int B, N, P, KC;
  const float *b0, *b1;  // bias: mean (LRT, plain) or sampled (Flipout); sigma_b (LRT)
  NoiseRef eps, drop;    // LRT eps [B, N * P]; dropout keep decisions [B, N, P] (plain mode)
  float keep;
  const float* sout;     // Flipout s_out [B, N]
  float* act;            // [B * P, N] after ReLU and dropout
  float* rbuf;           // LRT: eps / (2 sd) [B * P, N]
  int* status;
};
template <int MODE>
__global__ void __launch_bounds__(128, 1) tc3_fwd_kernel(const Tc3FwdArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  constexpr bool DUAL = MODE != TT_PLAIN;
  const int mt = blockIdx.x, ns = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t tmem = tl_fwd_mainloop<MODE>(smem, a.a0, a.a1, a.w0, a.w1, a.KC, mt, ns, a.status);
  const int row = warp * 32 + lane, m = mt * 128 + row, N = a.N;
  const bool live = m < a.B * a.P;
  const int b = live ? m / a.P : 0, pos = m - b * a.P;
  const uint32_t la = tmem + ((uint32_t)(warp * 32) << 16);
#pragma unroll 1
  for (int g = 0; g < TL_NS / 8; ++g) {
    const int n0 = ns * TL_NS + g * 8;
    if (n0 >= N) break;  // conv1: columns 16..31 of the slice are padding
    float v0[8], v1[8];
    tmem_ld8(la + g * 8, v0);
    if (DUAL) tmem_ld8(la + TL_NS + g * 8, v1);
    tmem_ld_wait();
    if (!live) continue;
    const long long e0 = (long long)m * N + n0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int n = n0 + j;
      float pre;
      if (MODE == BRL_MODE_LRT) {
        const float sb = a.b1[n];
        float var = fmaf(sb, sb, v1[j]);
        if (var < 0.f) var += fabsf(var) + 1e-6f;
        const float sd = sqrtf(var), e = gnoise_normal(a.eps, 0, b, a.B, N * a.P, n * a.P + pos);
        pre = fmaf(sd, e, v0[j] + a.b0[n]);
        a.rbuf[e0 + j] = sd > 0.f ? e / (2.0f * sd) : 0.f;
      } else if (MODE == BRL_MODE_FLIPOUT) {
        pre = v0[j] + v1[j] * a.sout[(long long)b * N + n] + a.b0[n];
      } else {
        pre = v0[j] + a.b0[n];
      }
      float o = fmaxf(pre, 0.f);
      if (MODE == TT_PLAIN && a.keep < 1.0f) o = gnoise_keep(a.drop, 0, b, a.B, N, a.P, n, pos, a.keep) ? o / a.keep : 0.f;
      a.act[e0 + j] = o;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 64);
}

// AvgPool((2,1)) of conv3's activation and the flatten c * 5 + t: the tail's features [B, 320]; thread = one feature
__global__ void tc3_pool_kernel(const float* __restrict__ act3, float* __restrict__ feat, int B) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * 320) return;
  const int b = i / 320, f = i - b * 320, c = f / 5, t = f - c * 5;
  const float* p = act3 + ((long long)b * 11 + 2 * t) * 64 + c;
  feat[i] = 0.5f * (p[0] + p[64]);
}

// activation backward of conv l: the gradient w.r.t. its output [B * P, N] (l = 2: from the features' gradient through the pool;
// l = 1, 0: col2im of conv l + 1's column gradients, the second path combined with conv l + 1's input -- 2 a (LRT) or s_in
// (Flipout) -- then through the pool in front of conv3 for l = 1); the ReLU / dropout gate comes from the stored activation.
// Rows the floor-mode pools drop (conv2 row 24, conv3 row 10) receive zero.  Thread = one (row, channel).
struct Tc3ActBwdArgs {
  int l, B, mode;
  float keep;              // dropout site behind conv l (plain mode)
  const float *src0, *src1;  // l = 2: d features [B, 320]; else conv l + 1's column gradients [B * P', K'] (mean / second path)
  const float* act;        // conv l's activation [B * P, N]
  const float* rb;         // LRT: conv l's eps / (2 sd)
  const float* sout;       // Flipout: conv l's s_out [B, N]
  const float* sin_next;   // Flipout: conv l + 1's s_in [B, N]
  float *d0, *d1;          // conv l's compact gradients [B * P, N]: pre-activation / second path
};
__global__ void tc3_bwd_act_kernel(const Tc3ActBwdArgs a) {
  const int l = a.l, N = tc3_n(l), P = tc3_p(l);
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= (long long)a.B * P * N) return;
  const int m = (int)(i / N), c = (int)(i - (long long)m * N), b = m / P, pos = m - b * P;
  const float av = a.act[i];
  float d = 0.f;
  if (l == 2) {
    if (pos < 10) d = 0.5f * a.src0[(long long)b * 320 + c * 5 + (pos >> 1)];
  } else {
    float s0 = 0.f, s1 = 0.f, x;
    if (l == 1) {  // conv3 reads pooled row t' = pos / 2 at (ci = c, kh) from its rows t' - kh
      if (pos < 24) {
        const int tp = pos >> 1;
#pragma unroll
        for (int kh = 0; kh < 2; ++kh) {
          const int t = tp - kh;
          if (t < 0 || t >= 11) continue;
          const long long e = ((long long)b * 11 + t) * 64 + c * 2 + kh;
          s0 += a.src0[e];
          if (a.mode != TT_PLAIN) s1 += a.src1[e];
        }
      }
      const float* p = a.act + ((long long)b * 25 + (pos & ~1)) * 32 + c;
      x = pos < 24 ? 0.5f * (p[0] + p[32]) : 0.f;  // the pooled input value (the second path's factor)
    } else {  // conv2 reads conv1's (oh, ow) at (ci = c, kh, kw = ow) from its rows oh - kh
      const int oh = pos / 10, ow = pos - oh * 10;
#pragma unroll
      for (int kh = 0; kh < 2; ++kh) {
        const int t = oh - kh;
        if (t < 0 || t >= 25) continue;
        const long long e = ((long long)b * 25 + t) * 320 + (c * 2 + kh) * 10 + ow;
        s0 += a.src0[e];
        if (a.mode != TT_PLAIN) s1 += a.src1[e];
      }
      x = av;
    }
    x = __half2float(__float2half_rn(x));  // as the forward operand
    const float dx = a.mode == BRL_MODE_LRT ? fmaf(2.0f * x, s1, s0) : a.mode == BRL_MODE_FLIPOUT ? fmaf(a.sin_next[b * N + c], s1, s0) : s0;
    d = (l == 1) ? (pos < 24 ? 0.5f * dx : 0.f) : dx;
  }
  // ReLU gate from the stored activation (with dropout a * m / keep: it gates, 1 / keep scales)
  const float g = av > 0.f ? (a.mode == TT_PLAIN ? d / a.keep : d) : 0.f;
  a.d0[i] = g;
  if (a.mode == BRL_MODE_LRT) a.d1[i] = g * a.rb[i];
  else if (a.mode == BRL_MODE_FLIPOUT) a.d1[i] = g * a.sout[b * N + c];
}
