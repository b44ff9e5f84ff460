// Level-fused tcgen05 training kernels of the Linear net (linear.py:44-55,66-70: Flatten 540 -> 256 -> 128 -> 128 -> 32 -> 2,
// ReLU behind the hidden layers, dropout sites behind hidden layers 0..3).  Included by brl_tc_train.cu, whose helpers it uses.
//
// Every hidden layer is a dense GEMM over 128-window M-tiles.  Operands are images in the fc layer's K-major chunk layout:
//     activation image of a layer input   [M-tile][K/8 chunks][128 windows][8 x 16 bit]   (K = 540 padded to 576 for x)
//     weight image of a layer             [N/32 slices][K/8 chunks][32 n][8 x 16 bit]     (an N-slice is contiguous)
// and the three contractions read them as the Inception fc kernels do:
//     forward           D[m, n] = sum_k a[m, k] W[n, k]      A K-major (activation image), B K-major (weight image)
//     input gradient    D[m, k] = sum_n g[m, n] W[n, k]      A K-major (gradient image),   B MN-major (weight image^T)
//     weight gradient   D[k, n] = sum_m a[m, k] g[m, n]      A MN-major (activation^T),    B MN-major (gradient^T)
// Modes (the dual contraction and its epilogue as in brl_tc_train.cu):
//     LRT      a * mu (fp16),  a^2 * sigma^2 (bf16)         relu(mean + b + eps * sqrt(var + sigma_b^2))
//     Flipout  a * mu (fp16),  (a . s_in) * (W - mu) (fp16)  relu(mean + pert . s_out + b_sampled)
//     plain    a * W (fp16): weight-sampling ELBO, HNN step (dropout keep decisions in the epilogue)
// Launches of one particle: window packing + weight packing (side stream), four forward launches (grid = M-tiles x 32-column
// slices; layer 3 leaves its raw sums to tt_tail_kernel, which runs layer 3's epilogue, the head, the likelihood and their
// backward), three input-gradient launches (layers 3, 2, 1; each fused with the activation backward of the layer below) on the
// critical chain, four weight-gradient launches on the side stream, each forked as soon as its layer's gradient exists.
// Gradients travel between kernels as compact fp32 [B, N] tensors (the tail's format); the consumers round them to bf16 while
// staging their operand image.

constexpr int TL_CH = 128 * 16;  // one 8-feature chunk of a 128-window M-tile
constexpr int TL_NS = 32;        // forward: output columns per CTA = rows of one weight-image slice
constexpr int TL_KS = 8;         // forward: chunks per pipeline stage (64 features, 4 MMA k-steps)
constexpr int TL_STAGES = 3;
constexpr int TL_XS = 64;        // input gradient: features per CTA
constexpr int TL_WS = 64;        // weight gradient: output columns per CTA (at most)
__host__ __device__ constexpr int tl_cin(int l) { return l == 0 ? 540 : l == 1 ? 256 : 128; }
__host__ __device__ constexpr int tl_kc(int l) { return l == 0 ? 72 : tl_cin(l) / 8; }  // chunks of the layer's input image
__host__ __device__ constexpr int tl_n(int l) { return l == 0 ? 256 : l == 3 ? 32 : 128; }
__host__ __device__ constexpr int tl_wimg(int l) { return tl_n(l) * tl_kc(l) * 16; }   // bytes of one weight image
constexpr int TL_PACK_END = 256 * 576 + 128 * 256 + 128 * 128 + 32 * 128;             // weight elements of the four layers

// ------------------------------------------------------------------------------------------------
// packing: windows -> layer-0 input images (once per particle); weights -> four images per layer (side stream)
// ------------------------------------------------------------------------------------------------
struct TlPackXArgs {
  const float* x;       // [B, 540]
  const float* sgn_in;  // Flipout s_in of layer 0 [B, 540]
  int B, mode;
  unsigned char* img[4];
};
__global__ void tl_packx_kernel(const TlPackXArgs a) {  // thread = 8 features of one window row
  const long long u = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const int nmt = (a.B + 127) >> 7;
  if (u >= (long long)nmt * 72 * 128) return;
  const int r = (int)(u & 127), c = (int)((u >> 7) % 72), mt = (int)((u >> 7) / 72), m = mt * 128 + r;
  float f[8], s[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int k = c * 8 + j;
    const bool on = m < a.B && k < 540;
    f[j] = on ? __half2float(__float2half_rn(a.x[(long long)m * 540 + k])) : 0.f;
    s[j] = a.mode == BRL_MODE_LRT ? f[j] * f[j] : (a.mode == BRL_MODE_FLIPOUT && on) ? f[j] * a.sgn_in[(long long)m * 540 + k] : 0.f;
  }
  const long long o = (long long)u * 16;  // u = (mt * 72 + c) * 128 + r: the image offset in 16-byte units
  *reinterpret_cast<uint4*>(a.img[0] + o) = pack_h8(f);
  *reinterpret_cast<uint4*>(a.img[1] + o) = pack_b8(f);
  if (a.mode == BRL_MODE_LRT) {
    *reinterpret_cast<uint4*>(a.img[2] + o) = pack_b8(s);
  } else if (a.mode == BRL_MODE_FLIPOUT) {
    *reinterpret_cast<uint4*>(a.img[2] + o) = pack_h8(s);
    *reinterpret_cast<uint4*>(a.img[3] + o) = pack_b8(s);
  }
}

struct TlPackWArgs {
  int mode;
  const float *mu, *second;  // second: sigma (LRT) or the weight draw (Flipout)
  long long w_off[4];
  unsigned char* w[4];       // fp16 mu | bf16 mu | bf16 sigma^2 or (W - mu) | fp16 (W - mu)
};
__global__ void tl_pack_w_kernel(const TlPackWArgs a) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= TL_PACK_END) return;
  int l = 0;
  while (j >= tl_n(l) * tl_kc(l) * 8) { j -= tl_n(l) * tl_kc(l) * 8; ++l; }
  const int K8 = tl_kc(l) * 8, cin = tl_cin(l), n = j / K8, k = j - n * K8;  // consecutive threads: consecutive k (coalesced reads)
  float m = 0.f, s = 0.f;
  // the parameter arrays are indexed through a switch: a dynamic index would copy them to local memory
  const long long w_off = l == 0 ? a.w_off[0] : l == 1 ? a.w_off[1] : l == 2 ? a.w_off[2] : a.w_off[3];
  unsigned char* w = l == 0 ? a.w[0] : l == 1 ? a.w[1] : l == 2 ? a.w[2] : a.w[3];
  if (k < cin) {
    const long long wi = w_off + (long long)n * cin + k;
    m = a.mu[wi];
    const float v = a.second[wi];
    s = a.mode == BRL_MODE_LRT ? v * v : a.mode == BRL_MODE_FLIPOUT ? v - m : 0.f;
  }
  const int o = (((n >> 5) * tl_kc(l) + (k >> 3)) * 32 + (n & 31)) * 16 + (k & 7) * 2, img = tl_wimg(l);
  *reinterpret_cast<__half*>(w + o) = __float2half_rn(m);
  *reinterpret_cast<__nv_bfloat16*>(w + img + o) = __float2bfloat16_rn(m);
  *reinterpret_cast<__nv_bfloat16*>(w + 2 * img + o) = __float2bfloat16_rn(s);
  *reinterpret_cast<__half*>(w + 3 * img + o) = __float2half_rn(s);
}

// ------------------------------------------------------------------------------------------------
// forward: one CTA = 32 output columns of one hidden layer for one M-tile; K streams through a 3-stage ring of 64-feature slabs
// ------------------------------------------------------------------------------------------------
constexpr int TLF_STG = 2 * TL_KS * TL_CH + 2 * TL_KS * 512;  // A | A2 | W0 | W1 of one slab
constexpr int TLF_BAR = TL_STAGES * TLF_STG, TLF_SMEM = TLF_BAR + 128;
struct TlFwdArgs {
  const unsigned char *a0, *a1;  // input images: fp16 a; bf16 a^2 (LRT) or fp16 a * s_in (Flipout)
  const unsigned char *w0, *w1;  // weight images: fp16 mu; bf16 sigma^2 (LRT) or fp16 (W - mu) (Flipout)
  int B, N, KC, last;            // last: layer 3 -- raw sums to `part`, its epilogue runs in the tail
  const float *b0, *b1;          // bias: mean (LRT, plain) or sampled (Flipout); sigma_b (LRT)
  NoiseRef eps, drop;            // LRT eps [B, N]; dropout keep decisions behind the ReLU (plain mode)
  float keep;                    // keep probability of that site (1 = none)
  const float* sout;             // Flipout s_out [B, N]
  const float* sin_next;         // Flipout s_in of the next layer [B, N]
  unsigned char* out[4];         // the next layer's input images (same four roles as the inputs)
  float* rbuf;                   // LRT: eps / (2 sd) [B, N] for the backward pass
  float* part;                   // last: [2][B][N]
  int* status;
};
// the K loop shared by the forward kernels (tl_fwd_kernel, tc3_fwd_kernel): sets up the CTA's barriers and 64 TMEM columns, thread 0
// streams the slabs of M-tile `mt` / 32-column weight slice `ns` through the ring and issues the MMAs (mean path at column 0, the
// second path at column TL_NS); every thread returns the TMEM base once the accumulators are complete
template <int MODE>
__device__ __forceinline__ uint32_t tl_fwd_mainloop(unsigned char* smem, const unsigned char* a0, const unsigned char* a1,
                                                    const unsigned char* w0, const unsigned char* w1, int KC, int mt, int ns, int* status) {
  constexpr bool DUAL = MODE != TT_PLAIN;
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t sbase = smem_u32(smem), bfull = sbase + TLF_BAR, bempty = bfull + 8 * TL_STAGES, bdone = bempty + 8 * TL_STAGES;
  uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + TLF_BAR + 64);
  if (tid == 0) {
    for (int s = 0; s < TL_STAGES; ++s) { mbar_init(bfull + 8 * s, 1); mbar_init(bempty + 8 * s, 1); }
    mbar_init(bdone, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc(smem_u32(tslot), 64);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tslot;
  if (tid == 0) {  // producer and MMA issuer: slab `it` is loaded while slab `it - 2` is multiplied
    const int nslab = KC / TL_KS;
    const long long ao = (long long)mt * KC * TL_CH, wo = (long long)ns * KC * 512;
    for (int it = 0; it < nslab + TL_STAGES - 1; ++it) {
      if (it < nslab) {
        const int s = it % TL_STAGES;
        if (it >= TL_STAGES) mbar_wait(bempty + 8 * s, (it / TL_STAGES - 1) & 1, status, 60);
        const uint32_t st = sbase + s * TLF_STG, bar = bfull + 8 * s;
        mbar_expect_tx(bar, (DUAL ? 2 : 1) * (TL_KS * TL_CH + TL_KS * 512));
        bulk_g2s(st, a0 + ao + (long long)it * TL_KS * TL_CH, TL_KS * TL_CH, bar);
        bulk_g2s(st + 2 * TL_KS * TL_CH, w0 + wo + it * TL_KS * 512, TL_KS * 512, bar);
        if (DUAL) {
          bulk_g2s(st + TL_KS * TL_CH, a1 + ao + (long long)it * TL_KS * TL_CH, TL_KS * TL_CH, bar);
          bulk_g2s(st + 2 * TL_KS * TL_CH + TL_KS * 512, w1 + wo + it * TL_KS * 512, TL_KS * 512, bar);
        }
      }
      const int j = it - (TL_STAGES - 1);
      if (j >= 0) {
        const int s = j % TL_STAGES;
        mbar_wait(bfull + 8 * s, (j / TL_STAGES) & 1, status, 61);
        tc_fence_after();
        const uint32_t st = sbase + s * TLF_STG;
        for (int ks = 0; ks < TL_KS / 2; ++ks) {
          const uint32_t acc = (j | ks) != 0;
          umma(tmem, umma_desc(st + 2 * ks * TL_CH, TL_CH, 128), umma_desc(st + 2 * TL_KS * TL_CH + 2 * ks * 512, 512, 128),
               tt_idesc(TL_NS, 0, 0, 0), acc);
          if (DUAL)
            umma(tmem + TL_NS, umma_desc(st + TL_KS * TL_CH + 2 * ks * TL_CH, TL_CH, 128),
                 umma_desc(st + 2 * TL_KS * TL_CH + TL_KS * 512 + 2 * ks * 512, 512, 128),
                 tt_idesc(TL_NS, MODE == BRL_MODE_LRT ? 1 : 0, 0, 0), acc);
        }
        umma_commit(bempty + 8 * s);
      }
    }
    umma_commit(bdone);
  }
  mbar_wait(bdone, 0, status, 62);
  tc_fence_after();
  return tmem;
}

template <int MODE>
__global__ void __launch_bounds__(128, 1) tl_fwd_kernel(const TlFwdArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  constexpr bool DUAL = MODE != TT_PLAIN;
  const int mt = blockIdx.x, ns = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t tmem = tl_fwd_mainloop<MODE>(smem, a.a0, a.a1, a.w0, a.w1, a.KC, mt, ns, a.status);
  // ---- epilogue: thread = window row (TMEM lane), eight columns at a time
  const int row = warp * 32 + lane, m = mt * 128 + row, N = a.N;
  const bool live = m < a.B;
  const uint32_t la = tmem + ((uint32_t)(warp * 32) << 16);
#pragma unroll 1
  for (int g = 0; g < TL_NS / 8; ++g) {
    const int n0 = ns * TL_NS + g * 8;
    float v0[8], v1[8], o[8];
    tmem_ld8(la + g * 8, v0);
    if (DUAL) tmem_ld8(la + TL_NS + g * 8, v1);
    tmem_ld_wait();
    const long long e0 = (long long)m * N + n0;
    if (a.last) {
      if (live)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          a.part[e0 + j] = v0[j];
          if (DUAL) a.part[(long long)a.B * N + e0 + j] = v1[j];
        }
      continue;
    }
    float ev[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) ev[j] = 0.f;
    if (MODE == BRL_MODE_LRT && live) {  // element order e = n (one position): two Philox blocks of four normals
      if (a.eps.ptr) {
#pragma unroll
        for (int j = 0; j < 8; ++j) ev[j] = a.eps.ptr[e0 + j];
      } else {
        const NoiseKey k = noise_key(a.eps);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const float4 z = normal4(philox_block(k.seed, a.eps.kind, a.eps.site, k.sample0, k.window0 + m, (uint32_t)(n0 >> 2) + h));
          ev[4 * h] = z.x; ev[4 * h + 1] = z.y; ev[4 * h + 2] = z.z; ev[4 * h + 3] = z.w;
        }
      }
    }
    KeepBits kb = {};
    const bool drop = MODE == TT_PLAIN && a.keep < 1.0f;
    if (drop && live && !a.drop.ptr) {  // 8 of the 16 keep decisions of one Philox block (philox_keep, C = N, position 0)
      const NoiseKey dk = noise_key(a.drop);
      kb = keep_bits(philox_block_mask(dk.seed, a.drop.kind, a.drop.site, dk.sample0, dk.window0 + m, (uint32_t)(n0 >> 4)),
                     keep_threshold(a.keep));
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int n = n0 + j;
      float pre;
      if (MODE == BRL_MODE_LRT) {
        const float sb = a.b1[n];
        float var = fmaf(sb, sb, v1[j]);
        if (var < 0.f) var += fabsf(var) + 1e-6f;
        const float sd = sqrtf(var);
        pre = fmaf(sd, ev[j], v0[j] + a.b0[n]);
        if (live) a.rbuf[e0 + j] = sd > 0.f ? ev[j] / (2.0f * sd) : 0.f;
      } else if (MODE == BRL_MODE_FLIPOUT) {
        pre = v0[j] + (live ? v1[j] * a.sout[e0 + j] : 0.f) + a.b0[n];
      } else {
        pre = v0[j] + a.b0[n];
      }
      o[j] = live ? fmaxf(pre, 0.f) : 0.f;
      if (drop && live) {
        const bool kp = a.drop.ptr ? a.drop.ptr[e0 + j] != 0.f : keep_at(kb, (uint32_t)(n & 15));
        o[j] = kp ? o[j] / a.keep : 0.f;
      }
    }
    // the next layer's operand images (dead rows are written as zeros: they are K rows of the weight-gradient GEMMs)
    const long long off = (((long long)mt * (N / 8) + (n0 >> 3)) * 128 + row) * 16;
    const uint4 oh = pack_h8(o);
    float fr[8], s[8];
    unpack_h8(oh, fr);
    *reinterpret_cast<uint4*>(a.out[0] + off) = oh;
    *reinterpret_cast<uint4*>(a.out[1] + off) = pack_b8(fr);
    if (MODE == BRL_MODE_LRT) {
#pragma unroll
      for (int j = 0; j < 8; ++j) s[j] = fr[j] * fr[j];
      *reinterpret_cast<uint4*>(a.out[2] + off) = pack_b8(s);
    } else if (MODE == BRL_MODE_FLIPOUT) {
#pragma unroll
      for (int j = 0; j < 8; ++j) s[j] = live ? fr[j] * a.sin_next[e0 + j] : 0.f;
      *reinterpret_cast<uint4*>(a.out[2] + off) = pack_h8(s);
      *reinterpret_cast<uint4*>(a.out[3] + off) = pack_b8(s);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 64);
}

// compact fp32 gradient columns [c0, c0 + ncol) of an M-tile -> bf16 K-major image [ncol / 8 chunks][128 windows][16 B];
// (T * nthreads >= 128 * ncol / 8 items); with `sums`, every thread also adds the values it stages to its column sums
// (items tid + nthreads * t, t < T)
template <int T>
__device__ __forceinline__ void tl_grad_image(const float* __restrict__ d, unsigned char* img, int mt, int B, int N, int c0, int ncol,
                                              int tid, int nthreads, float (*sums)[8]) {
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const int i = tid + t * nthreads;
    if (i >= 128 * (ncol >> 3)) break;
    const int r = i & 127, c = i >> 7, m = mt * 128 + r;
    float v[8];
    if (m < B) {
      const float* p = d + (long long)m * N + c0 + c * 8;
      const float4 lo = *reinterpret_cast<const float4*>(p), hi = *reinterpret_cast<const float4*>(p + 4);
      v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w; v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = 0.f;
    }
    *reinterpret_cast<uint4*>(img + c * TL_CH + r * 16) = pack_b8(v);
    if (sums)
#pragma unroll
      for (int j = 0; j < 8; ++j) sums[t][j] += v[j];
  }
}

// ------------------------------------------------------------------------------------------------
// input gradient of hidden layer l (1..3) fused with the activation backward of layer l - 1: one CTA = 64 input features of
// one M-tile; writes layer l - 1's compact gradients d/d(pre-activation) and d/d(variance or perturbation path)
// ------------------------------------------------------------------------------------------------
constexpr int TLX_G0 = 0, TLX_G1 = 16 * TL_CH, TLX_W0 = 32 * TL_CH, TLX_W1 = TLX_W0 + 4 * 4096, TLX_BAR = TLX_W1 + 4 * 4096;
constexpr int TLX_SMEM = TLX_BAR + 64;
struct TlDxArgs {
  const float *g0, *g1;          // layer l's compact gradients [B, Nl]
  const unsigned char *w0, *w1;  // layer l's bf16 weight images (mu; sigma^2 or W - mu)
  const unsigned char* act;      // fp16 input image of layer l (= layer l - 1's stored activation)
  int B, Nl, KCl;                // KCl * 8 = layer l's input width
  const float* sin_;             // Flipout: layer l's s_in [B, KCl * 8]
  const float* rb;               // LRT: layer l - 1's eps / (2 sd)
  const float* sout;             // Flipout: layer l - 1's s_out
  float keep;                    // dropout site behind layer l - 1 (plain mode)
  float *d0, *d1;                // layer l - 1's compact gradients [B, KCl * 8]
  int raw;                       // 1: d0 / d1 receive the two GEMM results as they are (Conv-D3: col2im follows), no activation backward
  int* status;
};
template <int MODE>
__global__ void __launch_bounds__(256, 1) tl_dx_kernel(const TlDxArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  constexpr bool DUAL = MODE != TT_PLAIN;
  const int mt = blockIdx.x, xs = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem), bar_ld = sbase + TLX_BAR, bar_mma = bar_ld + 8;
  uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + TLX_BAR + 16);
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
  const int nsl = a.Nl / 32;
  if (tid == 0) {  // the eight chunks of this CTA's features from every 32-unit slice of the weight images
    mbar_expect_tx(bar_ld, (DUAL ? 2 : 1) * nsl * 4096);
    for (int s = 0; s < nsl; ++s) {
      const long long wo = ((long long)s * a.KCl + xs * 8) * 512;
      bulk_g2s(sbase + TLX_W0 + s * 4096, a.w0 + wo, 4096, bar_ld);
      if (DUAL) bulk_g2s(sbase + TLX_W1 + s * 4096, a.w1 + wo, 4096, bar_ld);
    }
  }
  tl_grad_image<8>(a.g0, smem + TLX_G0, mt, a.B, a.Nl, 0, a.Nl, tid, 256, nullptr);  // Nl <= 128: 16 chunks x 128 rows
  if (DUAL) tl_grad_image<8>(a.g1, smem + TLX_G1, mt, a.B, a.Nl, 0, a.Nl, tid, 256, nullptr);
  mbar_wait(bar_ld, 0, a.status, 63);
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    if (elect_one()) {
      for (int ks = 0; ks < a.Nl / 16; ++ks) {  // 16 units per k-step; B = the weight image read MN-major
        const uint32_t bo = (ks >> 1) * 4096 + (ks & 1) * 256;
        umma(tmem, umma_desc(sbase + TLX_G0 + 2 * ks * TL_CH, TL_CH, 128), umma_desc(sbase + TLX_W0 + bo, 128, 512),
             tt_idesc(TL_XS, 1, 0, 1), ks != 0);
        if (DUAL)
          umma(tmem + TL_XS, umma_desc(sbase + TLX_G1 + 2 * ks * TL_CH, TL_CH, 128), umma_desc(sbase + TLX_W1 + bo, 128, 512),
               tt_idesc(TL_XS, 1, 0, 1), ks != 0);
      }
      umma_commit(bar_mma);
    }
    __syncwarp();
  }
  mbar_wait(bar_mma, 0, a.status, 64);
  tc_fence_after();
  const int row = (warp & 3) * 32 + lane, half = warp >> 2, m = mt * 128 + row, cin = a.KCl * 8;
  const uint32_t la = tmem + ((uint32_t)((warp & 3) * 32) << 16);
#pragma unroll 1
  for (int g = half * 4; g < half * 4 + 4; ++g) {
    float v0[8], v1[8], av[8];
    tmem_ld8(la + g * 8, v0);
    if (DUAL) tmem_ld8(la + TL_XS + g * 8, v1);
    tmem_ld_wait();
    if (m >= a.B) continue;
    const int k0 = xs * TL_XS + g * 8;
    if (a.raw) {
      const long long r0 = (long long)m * cin + k0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        a.d0[r0 + j] = v0[j];
        if (DUAL) a.d1[r0 + j] = v1[j];
      }
      continue;
    }
    unpack_h8(*reinterpret_cast<const uint4*>(a.act + (((long long)mt * a.KCl + (k0 >> 3)) * 128 + row) * 16), av);
    const long long e0 = (long long)m * cin + k0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float dA = v0[j];
      if (MODE == BRL_MODE_LRT) dA = fmaf(2.0f * av[j], v1[j], dA);
      else if (MODE == BRL_MODE_FLIPOUT) dA = fmaf(a.sin_[e0 + j], v1[j], dA);
      // ReLU gate from the stored activation (with dropout a * m / keep: it gates, 1 / keep scales)
      const float d = av[j] > 0.f ? (MODE == TT_PLAIN ? dA / a.keep : dA) : 0.f;
      a.d0[e0 + j] = d;
      if (MODE == BRL_MODE_LRT) a.d1[e0 + j] = d * a.rb[e0 + j];
      else if (MODE == BRL_MODE_FLIPOUT) a.d1[e0 + j] = d * a.sout[e0 + j];
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 128);
}

// ------------------------------------------------------------------------------------------------
// weight gradient of hidden layer l: one CTA = 128 input features x (up to) 64 output columns, K = the M-tiles
// [blockIdx.z * mt_per, + mt_per); results as plain stores (one CTA per output: Linear) or atomics into the zeroed accumulators
// (the M-tiles split over gridDim.z CTAs: Conv-D3).  The CTAs of feature tile 0 also write the bias sums.
// ------------------------------------------------------------------------------------------------
constexpr int TLW_A0 = 0, TLW_A1 = 16 * TL_CH, TLW_G0 = 32 * TL_CH, TLW_G1 = 40 * TL_CH, TLW_SUM = 48 * TL_CH,
              TLW_BAR = TLW_SUM + 512, TLW_SMEM = TLW_BAR + 64;
struct TlDwArgs {
  const unsigned char *a0, *a1;  // bf16 input images of layer l: a; a^2 (LRT) or a * s_in (Flipout)
  const float *g0, *g1;          // compact gradients [B, N]
  int B, N, KC, cin, nsl;
  int mt_per, atomic;
  float *gw0, *gw1;
  long long w_off, b_off;
  int* status;
};
template <int MODE>
__global__ void __launch_bounds__(256, 1) tl_dw_kernel(const TlDwArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  constexpr bool DUAL = MODE != TT_PLAIN;
  const int kt = blockIdx.x, n0 = blockIdx.y * a.nsl, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem), bar_ld = sbase + TLW_BAR, bar_mma = bar_ld + 8;
  uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + TLW_BAR + 16);
  float* sums = reinterpret_cast<float*>(smem + TLW_SUM);  // [2][64] bias sums
  if (tid == 0) {
    mbar_init(bar_ld, 1);
    mbar_init(bar_mma, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid < 128) sums[tid] = 0.f;
  if (warp == 0) tmem_alloc(smem_u32(tslot), 128);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tslot;
  // the last feature tile of layer 0 holds 8 chunks: features beyond them are accumulator rows nobody reads
  const int nch = min(16, a.KC - kt * 16), mt0 = blockIdx.z * a.mt_per, mt1 = min((a.B + 127) / 128, mt0 + a.mt_per);
  float bs0[4][8], bs1[4][8];
#pragma unroll
  for (int t = 0; t < 4; ++t)
#pragma unroll
    for (int j = 0; j < 8; ++j) bs0[t][j] = bs1[t][j] = 0.f;
  uint32_t ph = 0;
  for (int mt = mt0; mt < mt1; ++mt) {
    if (tid == 0) {
      const long long ao = ((long long)mt * a.KC + kt * 16) * TL_CH;
      mbar_expect_tx(bar_ld, (DUAL ? 2 : 1) * nch * TL_CH);
      bulk_copy_chunked(sbase + TLW_A0, a.a0 + ao, nch * TL_CH, bar_ld);
      if (DUAL) bulk_copy_chunked(sbase + TLW_A1, a.a1 + ao, nch * TL_CH, bar_ld);
    }
    tl_grad_image<4>(a.g0, smem + TLW_G0, mt, a.B, a.N, n0, a.nsl, tid, 256, bs0);  // nsl <= 64: 8 chunks x 128 rows
    if (DUAL) tl_grad_image<4>(a.g1, smem + TLW_G1, mt, a.B, a.N, n0, a.nsl, tid, 256, bs1);
    mbar_wait(bar_ld, ph, a.status, 65);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
      if (elect_one()) {
        for (int k = 0; k < 8; ++k) {  // 16 windows per k-step; both operands MN-major
          const uint32_t acc = (mt != mt0) | (k != 0);
          umma(tmem, umma_desc(sbase + TLW_A0 + k * 256, 128, TL_CH), umma_desc(sbase + TLW_G0 + k * 256, 128, TL_CH),
               tt_idesc(a.nsl, 1, 1, 1), acc);
          if (DUAL)
            umma(tmem + TL_WS, umma_desc(sbase + TLW_A1 + k * 256, 128, TL_CH), umma_desc(sbase + TLW_G1 + k * 256, 128, TL_CH),
                 tt_idesc(a.nsl, 1, 1, 1), acc);
        }
        umma_commit(bar_mma);
      }
      __syncwarp();
    }
    mbar_wait(bar_mma, ph, a.status, 66);
    tc_fence_after();
    ph ^= 1;
    __syncthreads();  // the next M-tile's copies and operand writes overwrite what these MMAs read
  }
  const int k = kt * 128 + (warp & 3) * 32 + lane, half = warp >> 2;
  const uint32_t la = tmem + ((uint32_t)((warp & 3) * 32) << 16);
#pragma unroll 1
  for (int g = half; g < a.nsl / 8; g += 2) {
    float v0[8], v1[8];
    tmem_ld8(la + g * 8, v0);
    if (DUAL) tmem_ld8(la + TL_WS + g * 8, v1);
    tmem_ld_wait();
    if (k < a.cin)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const long long wi = a.w_off + (long long)(n0 + g * 8 + j) * a.cin + k;
        if (a.atomic) {
          atomicAdd(a.gw0 + wi, v0[j]);
          if (DUAL) atomicAdd(a.gw1 + wi, v1[j]);
        } else {
          a.gw0[wi] = v0[j];
          if (DUAL) a.gw1[wi] = v1[j];
        }
      }
  }
  if (kt == 0) {  // bias: column sums of the staged gradients (a warp's items share their chunk: t-th chunk = (tid >> 7) + 2 t)
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int c = (tid >> 7) + 2 * t;
      if (c >= a.nsl / 8) break;
      const float s0 = warp_sum8(bs0[t], lane), s1 = DUAL ? warp_sum8(bs1[t], lane) : 0.f;
      if ((lane & 3) == 0) {
        atomicAdd(&sums[c * 8 + ((lane >> 2) & 7)], s0);
        if (DUAL) atomicAdd(&sums[64 + c * 8 + ((lane >> 2) & 7)], s1);
      }
    }
    __syncthreads();
    if (tid < a.nsl) {
      const float s1 = MODE == BRL_MODE_LRT ? sums[64 + tid] : sums[tid];  // Flipout: the sampled bias
      if (a.atomic) {
        atomicAdd(a.gw0 + a.b_off + n0 + tid, sums[tid]);
        if (DUAL) atomicAdd(a.gw1 + a.b_off + n0 + tid, s1);
      } else {
        a.gw0[a.b_off + n0 + tid] = sums[tid];
        if (DUAL) a.gw1[a.b_off + n0 + tid] = s1;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 128);
}
