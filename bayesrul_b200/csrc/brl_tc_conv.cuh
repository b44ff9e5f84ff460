// tcgen05 conv-stack kernel (included by brl_tc.cu after the PTX wrappers and geometry constants).
//
// One persistent CTA per SM, 20 warps (16 epilogue + 3 issuers + loader).  Warps 16..19 are the ISSUERS (phase B + bulk copies of slot 0 / 1, phases C + A of slot
// 0 / 1; converged, one elected lane issues).  Warps 0..15 are EPILOGUE warps (TMEM -> registers -> fp16 -> shared memory / feature
// tensor).  Two tile SLOTS are in flight per CTA (a tile = 128 rows = 4 windows x 32 rows, warp quadrant = window,
// lane = time step); each slot owns a 66 KB activation region, 256 TMEM columns and its own mbarriers.  All sixteen
// epilogue warps work on ONE slot at a time (thread = row x column quarter) and alternate between the slots, so the
// MMAs of one slot always run underneath the epilogue of the other one; there is no CTA- or group-wide barrier in
// the steady state -- warps only wait on "MMA done" mbarriers and arrive on "operands ready" mbarriers.
//
// Activation region of a slot (K-major, no swizzle: [8-channel chunk][132 rows][16 B]):
//   M1  16 chunks  module-1 output, 4 branches x 32 channels (27 real + const-1 channel + zeros)
//   M1P 16 chunks  MaxPool1d(3,1,1)(M1)  -- produced in the phase-A epilogue with warp shuffles (row = lane)
//   T2 / T3 (8 + 8 chunks) alias M1   (written after the MMAs reading M1 have completed)
//   X / XP  (3 + 3 chunks) alias M1P  (fp16 chunk images of the windows / their max-pool, prepared once per batch by
//                                      tc_packx_kernel and bulk-copied in; the 4th K chunk is a shared zero chunk
//                                      reached through the descriptor's leading-dimension offset)
// TMEM columns of a slot: phase A -> 128..255, phase B -> 0..175, phase C -> 0..127, so the next tile's phase A runs
// while the phase-C epilogue of the current one is still reading.
// MMA count per tile is kept low because every M=128 MMA re-reads its 4 KB A slice from shared memory whatever N is:
//   phase A  convs that share an input shift share one MMA (N = 96 / 64 / 32 for |shift| = 0 / 1 / 2)      -> 16 MMAs
//   phase B  [b1 | b2a | b3a] as one N = 144 GEMM over M1, b4 (N = 32) over pooled M1                          -> 16 MMAs
//   phase C  all taps of a k3 / k5 conv are concatenated along N (N = 48 / 80, un-shifted A) and the tap shift is
//            applied afterwards in registers: out[t] = sum_tap P_tap[t + tap - pad] via rotating shuffles       ->  8 MMAs
// Biases ride in the MMAs: input feature 18 is a constant 1 whose weight row (centre tap only) holds the bias;
// conv1's column 27 reproduces the constant into M1 (and, pooled, into M1P) for the module-2 1x1 convs.
#pragma once

struct ConvArgs {
  const unsigned char* ximg;  // [2 * npair][X0 X1 X2 XP0 XP1 XP2][132 rows][16 B]  (tc_packx_kernel)
  const unsigned char* blob;  // [images][BLOB_BYTES]: MC sample s reads image (s + img_phase) / img_per
  long long blob_stride;      // BLOB_BYTES or 0
  int img_per, img_phase;     // 1, 0: one image per sample; S, phase: one image per ensemble member of S samples
  unsigned char* feat;        // row-major [S][ntile128 * 128 windows][10 chunks][30 steps][8 fp16] (= [.., 2400] for the fc GEMM)
  int B, S, ntile4, ntile128;
  float keep4;                // dropout keep of the branch sites (1 = off)
  NoiseRef drop[12];
  // native dropout masks: the seven Philox round keys (the same for every thread: they ride in the kernel parameters, i.e. the
  // constant bank, instead of being re-derived by two adds per round per block), the sample / window origin of the key and
  // one bit per site that has an injected mask instead
  uint32_t rk[14];
  uint32_t sample0, window0, inj_mask;
  uint32_t keepT2;            // keep_threshold(keep4) in both 16-bit lanes
  int* status;
  long long* trace;  // debug: CTA 0 time stamps, [16 items][64 slots] (nullptr = off)
};

// fp32 windows -> fp16 chunk images of a tile: X (features 0..17, const 1 at 18) and XP = MaxPool1d(3,1,1)(X)
__global__ void tc_packx_kernel(const float* __restrict__ x, unsigned char* __restrict__ ximg, int B, int ntiles) {
  const long long u = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (u >= (long long)ntiles * 384) return;
  const int tile = (int)(u / 384), v = (int)(u % 384), c = v >> 7, r = v & 127;
  const int tt = r & 31, gw = tile * 4 + (r >> 5);
  float f[8], pm[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) f[j] = pm[j] = 0.f;
  if (tt < 30 && gw < B) {
    const float* px = x + (long long)gw * 540 + tt * 18 + c * 8;
    const int nf = c < 2 ? 8 : 2;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (j < nf) {
        const float v0 = __half2float(__float2half_rn(px[j]));
        float m = v0;
        if (tt > 0) m = fmaxf(m, __half2float(__float2half_rn(px[j - 18])));
        if (tt < 29) m = fmaxf(m, __half2float(__float2half_rn(px[j + 18])));
        f[j] = v0;
        pm[j] = m;
      }
    }
    if (c == 2) f[2] = pm[2] = 1.0f;  // feature 18 = 1: carries the biases
  }
  unsigned char* dst = ximg + (long long)tile * XIMG_TILE_BYTES + c * CS + (ROW0 + r) * 16;
  *reinterpret_cast<uint4*>(dst) = make_uint4(pack_h2(f[0], f[1]), pack_h2(f[2], f[3]), pack_h2(f[4], f[5]), pack_h2(f[6], f[7]));
  *reinterpret_cast<uint4*>(dst + 3 * CS) =
      make_uint4(pack_h2(pm[0], pm[1]), pack_h2(pm[2], pm[3]), pack_h2(pm[4], pm[5]), pack_h2(pm[6], pm[7]));
  if (r < 2 || r >= 126) {  // the zero pad rows above / below the tile travel with the image (one bulk copy per tile)
    const int pr = r < 2 ? r : r + 4;
    unsigned char* pd = ximg + (long long)tile * XIMG_TILE_BYTES + c * CS + pr * 16;
    *reinterpret_cast<uint4*>(pd) = make_uint4(0, 0, 0, 0);
    *reinterpret_cast<uint4*>(pd + 3 * CS) = make_uint4(0, 0, 0, 0);
  }
}

template <bool BIAS, int N>
__device__ __forceinline__ void act_plain(float (&v)[N], const float* bias) {
#pragma unroll
  for (int j = 0; j < N; ++j) v[j] = fmaxf(BIAS ? v[j] + bias[j] : v[j], 0.f);
}
// Injected dropout masks (parity tests): ReLU (+bias) and the mask of site `layer` on N fp32 accumulator columns = channels
// ch0.. of a site with `nvalid` channels, at time step t.  The 1 / keep scale of inverted dropout is NOT applied here: it is folded
// into the weights of the layer that reads the activation (tc_pack_kernel), where it costs nothing.
template <bool BIAS, int N>
__device__ __forceinline__ void act_injected(float (&v)[N], const float* bias, bool live, const ConvArgs& a, int layer, int s, int gw,
                                             int t, int ch0, int nvalid) {
#pragma unroll
  for (int j = 0; j < N; ++j) v[j] = fmaxf(BIAS ? v[j] + bias[j] : v[j], 0.f);
  if (live) {
    const float* m = a.drop[layer].ptr + ((long long)s * a.B + gw) * (nvalid * 30) + t;
#pragma unroll
    for (int j = 0; j < N; ++j)
      if (ch0 + j < nvalid) v[j] = m[(ch0 + j) * 30] != 0.f ? v[j] : 0.f;
  }
}
// Philox4x32-7 with the round keys read from the kernel parameters (bit-identical to brl_philox.cuh: philox_block_mask)
__device__ __forceinline__ uint4 philox7_rk(const ConvArgs& a, uint32_t block, uint32_t window, uint32_t sample, uint32_t site) {
  uint4 c = make_uint4(block, window, sample, (KIND_DROPOUT << 24) | site);
#pragma unroll
  for (int r = 0; r < 7; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ a.rk[2 * r], lo1, hi0 ^ c.w ^ a.rk[2 * r + 1], lo0);
  }
  return c;
}
// Native dropout masks work on the PACKED halves: the keep decisions of a channel pair are the two 16-bit lanes of one packed-half
// compare (brl_philox.cuh: keep_pair), so a pair is masked by ONE `and` behind the ReLU-and-pack convert.  One Philox block per 16
// channels; N = 8 uses the half of the block selected by ch0 (the neighbouring thread uses the other half).  Channels >= nvalid
// (zero columns and conv1's constant-1 column that carries the next module's biases) are not masked.  No 1 / keep scale (see above).
// ALLVALID: every channel ch0 .. ch0 + N - 1 is a real channel of the site (module-2 sites), so the nvalid tests fold away.
template <bool BIAS, int N, bool ALLVALID = false>
__device__ __forceinline__ void act_drop_packed(float (&v)[N], const float* bias, bool live, const ConvArgs& a, int layer, int s, int gw,
                                                int t, int ch0, int nvalid, uint32_t (&h)[N / 2]) {
  if (BIAS) {
#pragma unroll
    for (int j = 0; j < N; ++j) v[j] += bias[j];
  }
  const uint32_t e0 = (uint32_t)t * (uint32_t)((nvalid + 15) & ~15) + (uint32_t)ch0;
  // dead rows (time steps 30 / 31, windows >= B) must store zeros: with threshold 0 every decision is "drop"; the channels >= nvalid that
  // the masks below force to "keep" are exact zeros in a dead row anyway (no input, no tap shift reaches conv1's constant column)
  KeepBits kb = keep_bits_packed(philox7_rk(a, e0 >> 4, a.window0 + gw, a.sample0 + s, (uint32_t)layer), live ? a.keepT2 : 0u);
  if (N < 16 && (e0 & 8u)) {  // upper half of the block (warp-uniform): channel pairs 4..7 move to 0..3
    kb.ev[0] = kb.ev[2]; kb.ev[1] = kb.ev[3]; kb.od[0] = kb.od[2]; kb.od[1] = kb.od[3];
  }
#pragma unroll
  for (int p = 0; p < N / 2; ++p) {
    uint32_t m = keep_pair(kb, p);
    if (!ALLVALID) {
      if (ch0 + 2 * p + 1 >= nvalid) m |= 0xFFFF0000u;
      if (ch0 + 2 * p >= nvalid) m = 0xFFFFFFFFu;
    }
    h[p] = pack_relu_h2(v[2 * p], v[2 * p + 1]) & m;
  }
}
__device__ __forceinline__ uint4 pack8(const float* v, bool live) {
  uint4 r = make_uint4(pack_h2(v[0], v[1]), pack_h2(v[2], v[3]), pack_h2(v[4], v[5]), pack_h2(v[6], v[7]));
  if (!live) r = make_uint4(0, 0, 0, 0);
  return r;
}
__device__ __forceinline__ uint32_t hmax2u(uint32_t a, uint32_t b) {
  __half2 r = __hmax2(*reinterpret_cast<__half2*>(&a), *reinterpret_cast<__half2*>(&b));
  return *reinterpret_cast<uint32_t*>(&r);
}
// Rows of a window are the lanes of a warp and lanes 30 / 31 are dead rows that hold exact zeros, so a ROTATING
// shuffle implements both the zero padding of the tap shifts and the -inf padding of the max-pool (values >= 0).
__device__ __forceinline__ uint32_t pool3(uint32_t v, int lane) {
  const uint32_t up = __shfl_sync(0xffffffffu, v, (lane + 31) & 31), dn = __shfl_sync(0xffffffffu, v, (lane + 1) & 31);
  return hmax2u(v, hmax2u(up, dn));
}
__device__ __forceinline__ uint4 pool3x4(uint4 v, int lane) {
  return make_uint4(pool3(v.x, lane), pool3(v.y, lane), pool3(v.z, lane), pool3(v.w, lane));
}
__device__ __forceinline__ float shf(float v, int src_lane) { return __shfl_sync(0xffffffffu, v, src_lane); }
// ReLU + fp16 pack of 8 accumulator columns without bias / dropout: convert first, clamp on packed halves
__device__ __forceinline__ uint4 relu_pack8(const float* v, bool live) {
  uint32_t r[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) r[j] = live ? pack_relu_h2(v[2 * j], v[2 * j + 1]) : 0u;
  return make_uint4(r[0], r[1], r[2], r[3]);
}
// 16 accumulator columns -> two 16-byte fp16 chunks (ReLU, optional dropout of site `layer`)
template <bool DROP, bool ALLVALID = false>
__device__ __forceinline__ void finish16(float (&v)[16], bool live, const ConvArgs& a, int layer, int s, int gw, int t,
                                         int ch0, int nvalid, uint4& lo, uint4& hi) {
  if (DROP) {
    if ((a.inj_mask >> layer) & 1u) {
      act_injected<false, 16>(v, nullptr, live, a, layer, s, gw, t, ch0, nvalid);
      lo = pack8(v, live);
      hi = pack8(v + 8, live);
    } else {
      uint32_t h[8];
      act_drop_packed<false, 16, ALLVALID>(v, nullptr, live, a, layer, s, gw, t, ch0, nvalid, h);
      lo = make_uint4(h[0], h[1], h[2], h[3]);
      hi = make_uint4(h[4], h[5], h[6], h[7]);
    }
  } else {
    lo = relu_pack8(v, live);
    hi = relu_pack8(v + 8, live);
  }
}

#ifdef BRL_NOFEAT
#define BRL_FEAT_LIVE(x) ((x) && a.B < 0)
#else
#define BRL_FEAT_LIVE(x) (x)
#endif
#ifndef BRL_TRW0
#define BRL_TRW0 0
#define BRL_TRW1 15
#endif
constexpr int CONV_THREADS = 640;  // 16 epilogue warps + 4 issuer / loader warps (one per scheduler)
// mbarriers (byte offsets from OFF_BAR)
// every MMA phase commits twice (first / second accumulation chain), so a warp only waits for the columns it reads
constexpr int BAR_DONE_A = 0, BAR_DONE_A2 = 16, BAR_DONE_B = 32, BAR_DONE_B2 = 48, BAR_DONE_C = 64, BAR_DONE_C2 = 80,
              BAR_READY_A = 96, BAR_READY_B = 112, BAR_XFULL = 128, BAR_W = 144, BAR_WFREE = 152, BAR_TMEM_SLOT = 160,
              BAR_ABORT = 168;

template <bool DROP>
__global__ void __launch_bounds__(CONV_THREADS, 1) tc_conv_kernel(const ConvArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);  // broadcast: the compiler may treat it as warp-uniform
  const uint32_t bars = sbase + OFF_BAR;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + OFF_BAR + BAR_TMEM_SLOT);
  volatile int* abort_flag = reinterpret_cast<volatile int*>(smem + OFF_BAR + BAR_ABORT);

  // zero the activation regions (their pad rows stay zero for the whole kernel) and the shared zero chunk
  for (int i = tid; i < OFF_W / 16; i += CONV_THREADS) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
  for (int i = tid; i < CS / 16; i += CONV_THREADS) reinterpret_cast<uint4*>(smem + OFF_ZERO)[i] = make_uint4(0, 0, 0, 0);
  if (tid == 0) {
    *abort_flag = 0;
    for (int i = 0; i < 12; ++i) mbar_init(bars + 8 * i, 1);                // done A/A2/B/B2/C/C2 x 2 slots (tcgen05.commit)
    for (int i = 0; i < 4; ++i) mbar_init(bars + BAR_READY_A + 8 * i, 16);  // ready A / B x 2 slots: one arrival per epilogue warp
    for (int i = 0; i < 2; ++i) mbar_init(bars + BAR_XFULL + 8 * i, 1);     // bulk copies of the window images
    mbar_init(bars + BAR_W, 1);                                             // bulk copy of the weight image
    mbar_init(bars + BAR_WFREE, 16);                                        // all warps are done with the old weights
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), 512);
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  const int npair = (a.ntile4 + 1) >> 1;
  const long long total = (long long)a.S * npair;
  const long long per = (total + gridDim.x - 1) / gridDim.x;
  const long long beg = per * blockIdx.x, end = min(total, beg + per);

  if (warp >= 16) {
    // ======================================= ISSUERS / LOADERS ====================================
    // A tcgen05.mma issue blocks while the tensor pipe is busy, and a blocked issuer slows every other warp of its
    // scheduler, so the MMA stream is spread evenly over the four schedulers:
    //   warp 16 + k : phase B of slot k, then (its MMAs done = M1P space dead) the bulk copy of the slot's next window
    //                 images; warp 16 also copies the next MC sample's weight image
    //   warp 18 + k : phase C of slot k followed by phase A of the slot's next tile
    // Each warp runs converged (waits included) and one elected lane issues, so descriptors and addresses stay in
    // uniform registers (a lane-0-only branch costs ~80 cycles per tcgen05.mma).
    if (beg < end) {
      bool ok = true;
      const int k = warp & 1;  // slot
      const uint32_t rb = sbase + k * G_BYTES, tm = tmem + k * 256;
      auto tr = [&](long long it, int slot) {
        if (a.trace && blockIdx.x == 0 && lane == 0 && it - beg < 16) a.trace[(it - beg) * 128 + slot] = clock64();
      };
      if (warp < 18) {
        // phase B: module-2 1x1 convs: [b1 | b2a | b3a] (N = 144) on M1, b4 (N = 32) on pooled M1
        const uint64_t dWB1 = umma_desc(sbase + OFF_W + WI_B1, 2304, 128);
        const uint64_t dWB4 = umma_desc(sbase + OFF_W + WI_B4, 512, 128);
        const uint64_t dM1 = umma_desc(rb + R_M1 + ROW0 * 16, CS, 128), dM1P = umma_desc(rb + R_M1P + ROW0 * 16, CS, 128);
        uint32_t rph = 0u, fph = 0u;
        const uint64_t pol = l2_policy_evict_last();
        auto load_w = [&](int s) {
          if (elect_one()) {
            const unsigned char* src = a.blob + (long long)((s + a.img_phase) / a.img_per) * a.blob_stride;
            mbar_expect_tx(bars + BAR_W, CONV_IMG);
            for (int o = 0; o < CONV_IMG; o += 16384) bulk_g2s_hint(sbase + OFF_W + o, src + o, min(16384, CONV_IMG - o), bars + BAR_W, pol);
          }
          __syncwarp();
        };
        auto load_x = [&](int pair) {  // one bulk copy: X0 X1 X2 XP0 XP1 XP2 incl. their pad rows
          if (elect_one()) {
            const unsigned char* src = a.ximg + (long long)(pair * 2 + k) * XIMG_TILE_BYTES;
            mbar_expect_tx(bars + BAR_XFULL + 8 * k, XIMG_TILE_BYTES);
            bulk_g2s_hint(rb + R_X, src, XIMG_TILE_BYTES, bars + BAR_XFULL + 8 * k, pol);
          }
          __syncwarp();
        };
        int s = (int)(beg / npair), pair = (int)(beg % npair);
        load_x(pair);
        if (k == 0) load_w(s);
        for (long long it = beg; it < end && ok; ++it) {
          ok = mbar_wait_warp(bars + BAR_READY_A + 8 * k, rph, a.status, 2, abort_flag) && ok;
          tc_fence_after();
          tr(it, 40 + 2 * k);
          if (elect_one()) {
#pragma unroll
            for (int ks = 0; ks < 8; ++ks)
              umma(tm, dM1 + (uint64_t)((2 * ks * CS) >> 4), dWB1 + (uint64_t)((2 * ks * 2304) >> 4), umma_idesc(144), ks != 0);
            umma_commit(bars + BAR_DONE_B + 8 * k);
#pragma unroll
            for (int ks = 0; ks < 8; ++ks)
              umma(tm + 144, dM1P + (uint64_t)((2 * ks * CS) >> 4), dWB4 + (uint64_t)((2 * ks * 512) >> 4), umma_idesc(32), ks != 0);
            umma_commit(bars + BAR_DONE_B2 + 8 * k);
          }
          __syncwarp();
          tr(it, 41 + 2 * k);
          if (it + 1 < end) {
            const bool reload = pair + 1 == npair;
            if (reload) { pair = 0; ++s; } else ++pair;
            // the next tile's window images land in the M1P space as soon as the phase-B MMAs have read it
            ok = mbar_wait_warp(bars + BAR_DONE_B2 + 8 * k, rph, a.status, 9, abort_flag) && ok;
            load_x(pair);
            tr(it, 50 + k);
            if (reload && k == 0) {  // next MC sample: every warp has finished the old weights (MMAs complete, biases read)
              ok = mbar_wait_warp(bars + BAR_WFREE, fph, a.status, 4, abort_flag) && ok;
              fph ^= 1;
              load_w(s);
            }
          }
          rph ^= 1;
        }
      } else {
        const uint64_t dWC2 = umma_desc(sbase + OFF_W + WI_B2B, 48 * 16, 128);
        const uint64_t dWC3 = umma_desc(sbase + OFF_W + WI_B3B, 80 * 16, 128);
        const uint64_t dT2 = umma_desc(rb + R_T2 + ROW0 * 16, CS, 128), dT3 = umma_desc(rb + R_T3 + ROW0 * 16, CS, 128);
        uint32_t xph = 0u, wph = 0u, rph = 0u;
        // phase A: module 1.  TMEM cols (slot base + 128 +): conv5 0..31 | conv3 32..63 | conv1 64..95 | convpool 96..127
        auto issue_A = [&]() {
          ok = mbar_wait_warp(bars + BAR_XFULL + 8 * k, xph, a.status, 5, abort_flag) && ok;
          xph ^= 1;
          tc_fence_after();
          if (elect_one()) {
            // k-step 0 = chunks 0,1; k-step 1 = chunk 2 + the shared zero chunk (leading-dimension offset reaches it)
            const uint32_t zx = (uint32_t)(OFF_ZERO - (k * G_BYTES + R_X + 2 * CS)), zxp = (uint32_t)(OFF_ZERO - (k * G_BYTES + R_XP + 2 * CS));
            constexpr int shs[5] = {0, -1, 1, -2, 2}, nsh[5] = {96, 64, 64, 32, 32}, osh[5] = {0, 6144, 10240, 14336, 16384};
#pragma unroll
            for (int q = 0; q < 5; ++q)
#pragma unroll
              for (int ks = 0; ks < 2; ++ks)
                umma(tm + 128, umma_desc(rb + R_X + 2 * ks * CS + (ROW0 + shs[q]) * 16, ks ? zx : CS, 128),
                     umma_desc(sbase + OFF_W + WI_A + osh[q] + 2 * ks * nsh[q] * 16, nsh[q] * 16, 128), umma_idesc(nsh[q]), (q | ks) != 0);
            umma_commit(bars + BAR_DONE_A + 8 * k);
#pragma unroll
            for (int tp = 0; tp < 3; ++tp)
#pragma unroll
              for (int ks = 0; ks < 2; ++ks)
                umma(tm + 224, umma_desc(rb + R_XP + 2 * ks * CS + (ROW0 + tp - 1) * 16, ks ? zxp : CS, 128),
                     umma_desc(sbase + OFF_W + WI_A + 18432 + tp * 2048 + 2 * ks * 512, 512, 128), umma_idesc(32), (tp | ks) != 0);
            umma_commit(bars + BAR_DONE_A2 + 8 * k);
          }
          __syncwarp();
        };
        int pair = (int)(beg % npair);
        ok = mbar_wait_warp(bars + BAR_W, wph, a.status, 1, abort_flag) && ok;
        wph ^= 1;
        issue_A();
        for (long long it = beg; it < end && ok; ++it) {
          // phase C: b2b (k3 over T2) / b3b (k5 over T3): taps concatenated along N, shifts applied in the epilogue
          ok = mbar_wait_warp(bars + BAR_READY_B + 8 * k, rph, a.status, 3, abort_flag) && ok;  // T2 / T3 written, cols 128.. drained
          rph ^= 1;
          tc_fence_after();
          tr(it, 44 + 2 * k);
          if (elect_one()) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
              umma(tm, dT2 + (uint64_t)((2 * ks * CS) >> 4), dWC2 + (uint64_t)((2 * ks * 48 * 16) >> 4), umma_idesc(48), ks != 0);
            umma_commit(bars + BAR_DONE_C + 8 * k);
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
              umma(tm + 48, dT3 + (uint64_t)((2 * ks * CS) >> 4), dWC3 + (uint64_t)((2 * ks * 80 * 16) >> 4), umma_idesc(80), ks != 0);
            umma_commit(bars + BAR_DONE_C2 + 8 * k);
          }
          __syncwarp();
          tr(it, 45 + 2 * k);
          if (it + 1 < end) {  // phase A of the slot's next tile
            if (++pair == npair) {  // next MC sample: wait for the copy of the new weight image
              pair = 0;
              ok = mbar_wait_warp(bars + BAR_W, wph, a.status, 1, abort_flag) && ok;
              wph ^= 1;
            }
            issue_A();
            tr(it, 48 + k);
          }
        }
      }
    }
  } else {
    // ========================================== EPILOGUE ==========================================
    const int row = tid & 127, q = tid >> 7;  // q: column quarter (warp-uniform)
    const int wq = row >> 5, t = lane;
    const uint32_t rowoff = (uint32_t)(ROW0 + row) * 16;
    const uint32_t lane_base = tmem + ((uint32_t)(row & ~31) << 16);
    const float* sbias = reinterpret_cast<const float*>(smem + OFF_W + WI_BIAS);
    const int lm1 = (lane + 31) & 31, lm2 = (lane + 30) & 31, lp1 = (lane + 1) & 31, lp2 = (lane + 2) & 31;
    const int brA = q == 0 ? 2 : q == 1 ? 1 : q == 2 ? 0 : 3;  // TMEM column block q of phase A -> M1 channel group
    uint32_t ph = 0;
    bool ok = true;
    long long tr_it = beg;
    int tr_phase = 0;
    auto arrive_ready = [&](int bar, int k) {
      fence_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bars + bar + 8 * k);
      if (a.trace && blockIdx.x == 0 && lane == 0 && tr_it - beg < 16 && k == 0) a.trace[(tr_it - beg) * 128 + 64 + tr_phase * 16 + warp] = clock64();
    };
    const int trw = warp == BRL_TRW0 ? 0 : warp == BRL_TRW1 ? 18 : -1;
    auto tr = [&](long long it, int slot) {
      if (a.trace && blockIdx.x == 0 && trw >= 0 && lane == 0 && it - beg < 16) a.trace[(it - beg) * 128 + trw + slot] = clock64();
    };
    int s = (int)(beg / npair), pair = (int)(beg % npair);
    for (long long it = beg; it < end; ++it) {
      // ---- phase A epilogue: ReLU (+dropout) -> M1, MaxPool1d(3,1,1) -> M1P
      tr_it = it;
      tr_phase = 0;
#pragma unroll 1
      for (int k = 0; k < 2; ++k) {
        const int tile = pair * 2 + k, gw = tile * 4 + wq;
        const bool live = t < 30 && gw < a.B && tile < a.ntile4;
        unsigned char* reg = smem + k * G_BYTES;
        tr(it, 0 + 3 * k);
        ok = mbar_wait(bars + (q < 3 ? BAR_DONE_A : BAR_DONE_A2) + 8 * k, ph, a.status, 6, abort_flag) && ok;
        tc_fence_after();
        tr(it, 1 + 3 * k);
        float acc[2][16];
        tmem_ld16(lane_base + k * 256 + 128 + q * 32, acc[0]);
        tmem_ld16(lane_base + k * 256 + 128 + q * 32 + 16, acc[1]);
        tmem_ld_wait();
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          uint4 lo, hi;
          finish16<DROP>(acc[h], live, a, brA, s, gw, t, h * 16, 27, lo, hi);
          unsigned char* dst = reg + R_M1 + (brA * 4 + h * 2) * CS + rowoff;
          *reinterpret_cast<uint4*>(dst) = lo;
          *reinterpret_cast<uint4*>(dst + CS) = hi;
#ifdef BRL_POOL_SHFL
          *reinterpret_cast<uint4*>(dst + R_M1P) = pool3x4(lo, lane);  // R_M1P - R_M1 == 16 chunks
          *reinterpret_cast<uint4*>(dst + R_M1P + CS) = pool3x4(hi, lane);
#else
          // MaxPool1d(3,1,1) through shared memory: the neighbouring rows of a window are the neighbouring lanes' stores of the
          // two lines above (same warp: visible after __syncwarp); the rows next to a window (dead rows 30 / 31, pad rows) hold
          // zeros at all times, which is the -inf padding for values >= 0.  Four 16-byte loads instead of sixteen shuffles.
          __syncwarp();
          const uint4 z4 = make_uint4(0, 0, 0, 0);
          const uint4 plo = hmax4(lo, hmax4(*reinterpret_cast<const uint4*>(dst - 16), *reinterpret_cast<const uint4*>(dst + 16)));
          const uint4 phi = hmax4(hi, hmax4(*reinterpret_cast<const uint4*>(dst + CS - 16), *reinterpret_cast<const uint4*>(dst + CS + 16)));
          *reinterpret_cast<uint4*>(dst + R_M1P) = t < 30 ? plo : z4;  // R_M1P - R_M1 == 16 chunks
          *reinterpret_cast<uint4*>(dst + R_M1P + CS) = t < 30 ? phi : z4;
#endif
        }
        arrive_ready(BAR_READY_A, k);
        tr(it, 2 + 3 * k);
      }
      // ---- phase B epilogue: 11 groups of 16 columns: g0 = b1 -> feat ch 0..15 | g1..4 = b2a -> T2 | g5..8 = b3a -> T3 |
      //      g9,10 = b4 -> feat ch 48..79.  Quarter q takes T groups 1+2q, 2+2q and feat group {0, 9, 10, -}[q].
      tr_phase = 1;
#pragma unroll 1
      for (int k = 0; k < 2; ++k) {
        const int tile = pair * 2 + k, gw = tile * 4 + wq;
        const bool live = t < 30 && gw < a.B && tile < a.ntile4;
        unsigned char* reg = smem + k * G_BYTES;
        // feature row of window gw: chunk c of time step t at c * 480 + t * 16 -> a warp (one window, 30 steps) stores 480
        // contiguous bytes per chunk
        unsigned char* frow = a.feat + ((long long)s * a.ntile128 * 128 + gw) * FEAT_ROW_BYTES + t * 16;
        tr(it, 6 + 3 * k);
        ok = mbar_wait(bars + BAR_DONE_B + 8 * k, ph, a.status, 7, abort_flag) && ok;
        tc_fence_after();
        tr(it, 7 + 3 * k);
        const uint32_t la = lane_base + k * 256;
        float acc[3][16];
        tmem_ld16(la + (1 + 2 * q) * 16, acc[0]);
        tmem_ld16(la + (2 + 2 * q) * 16, acc[1]);
        if (q == 0) tmem_ld16(la, acc[2]);
        tmem_ld_wait();
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          unsigned char* dst = reg + R_T2 + (4 * q + 2 * h) * CS + rowoff;  // R_T3 == R_T2 + 8 chunks
          *reinterpret_cast<uint4*>(dst) = relu_pack8(acc[h], live);
          *reinterpret_cast<uint4*>(dst + CS) = relu_pack8(acc[h] + 8, live);
        }
        if (q == 1 || q == 2) {  // b4 columns come from the second accumulation chain of the phase
          ok = mbar_wait(bars + BAR_DONE_B2 + 8 * k, ph, a.status, 7, abort_flag) && ok;
          tc_fence_after();
          tmem_ld16(la + (q == 1 ? 9 : 10) * 16, acc[2]);
          tmem_ld_wait();
        }
        arrive_ready(BAR_READY_B, k);  // every TMEM column this thread needs is in registers: phase C may start now
        if (q < 3) {
          uint4 lo, hi;
          finish16<DROP, true>(acc[2], live, a, q == 0 ? 4 : 9, s, gw, t, q == 2 ? 16 : 0, q == 0 ? 16 : 32, lo, hi);
          const int fc = q == 0 ? 0 : q == 1 ? 6 : 8;
          if (BRL_FEAT_LIVE(live)) {
            st_global_cs(frow + fc * 480, lo);
            st_global_cs(frow + (fc + 1) * 480, hi);
          }
        }
        tr(it, 8 + 3 * k);
      }
      // ---- phase C epilogue: tap shifts in registers, bias, ReLU (+dropout) -> feat ch 16..47
#pragma unroll 1
      for (int k = 0; k < 2; ++k) {
        const int tile = pair * 2 + k, gw = tile * 4 + wq;
        const bool live = t < 30 && gw < a.B && tile < a.ntile4;
        // feature row of window gw: chunk c of time step t at c * 480 + t * 16 -> a warp (one window, 30 steps) stores 480
        // contiguous bytes per chunk
        unsigned char* frow = a.feat + ((long long)s * a.ntile128 * 128 + gw) * FEAT_ROW_BYTES + t * 16;
        tr(it, 12 + 3 * k);
        ok = mbar_wait(bars + (q < 2 ? BAR_DONE_C : BAR_DONE_C2) + 8 * k, ph, a.status, 8, abort_flag) && ok;
        tc_fence_after();
        tr(it, 13 + 3 * k);
        const uint32_t la = lane_base + k * 256;
        float out[8];
        if (q < 2) {  // b2b channels 8q..8q+7: out[t] = P0[t-1] + P1[t] + P2[t+1]
          float p[3][8];
#pragma unroll
          for (int tp = 0; tp < 3; ++tp) tmem_ld8(la + tp * 16 + q * 8, p[tp]);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 8; ++j) out[j] = shf(p[0][j], lm1) + p[1][j] + shf(p[2][j], lp1);
        } else {  // b3b channels 8(q-2)..: out[t] = sum_tap P_tap[t + tap - 2]
          float p[5][8];
#pragma unroll
          for (int tp = 0; tp < 5; ++tp) tmem_ld8(la + 48 + tp * 16 + (q - 2) * 8, p[tp]);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 8; ++j)
            out[j] = shf(p[0][j], lm2) + shf(p[1][j], lm1) + p[2][j] + shf(p[3][j], lp1) + shf(p[4][j], lp2);
        }
        tc_fence_before();
        if (DROP) {
          uint4 o4;
          if (!((a.inj_mask >> (q < 2 ? 6 : 8)) & 1u)) {
            uint32_t h[4];
            act_drop_packed<true, 8, true>(out, sbias + 304 + q * 8, live, a, q < 2 ? 6 : 8, s, gw, t, (q & 1) * 8, 16, h);
            o4 = make_uint4(h[0], h[1], h[2], h[3]);
          } else {
            act_injected<true, 8>(out, sbias + 304 + q * 8, live, a, q < 2 ? 6 : 8, s, gw, t, (q & 1) * 8, 16);
            o4 = pack8(out, true);
          }
          if (BRL_FEAT_LIVE(live)) st_global_cs(frow + (2 + q) * 480, o4);
        } else {
          act_plain<true, 8>(out, sbias + 304 + q * 8);
          if (BRL_FEAT_LIVE(live)) st_global_cs(frow + (2 + q) * 480, pack8(out, true));
        }
        tr(it, 14 + 3 * k);
      }
      if (++pair == npair) {
        pair = 0;
        ++s;
        if (it + 1 < end) {  // next MC sample: the issuer may now overwrite the weight image
          __syncwarp();
          if (lane == 0) mbar_arrive(bars + BAR_WFREE);
        }
      }
      ph ^= 1;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(*tmem_slot, 512);
}
