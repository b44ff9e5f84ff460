// tcgen05 predictive engine for the Conv-D3 net (nets/conv.py:47-61, 73-77): x.unsqueeze(1) [1,30,18] -> Conv2d(1,16,(5,9)) -> ReLU ->
// Conv2d(16,32,(2,10)) -> ReLU -> AvgPool((2,1)) -> Conv2d(32,64,(2,1)) -> ReLU -> AvgPool((2,1)) -> flatten 320 -> Linear(320,2) ->
// softplus + Threshold(1e-9) on both outputs; DET / weight-sampling forward without dropout.  Included by brl_tc.cu.
//
// A tile is FOUR windows: 128 rows = 4 windows x 32 rows (30 time steps + 2 dead rows), TMEM lane quadrant = window, lane = row, the
// shared-memory operands are K-major chunk images [8 k][132 rows][16 B] with two zero pad rows above and below (brl_tc.cu geometry), so
// that a kernel-height tap is a row shift of the A descriptor (as `padding = 'same'` is in the Inception engine).
//   conv1  the ten output columns ow form three groups (0-3, 4-7, 8-9); a group is ONE GEMM over the window slice x[:, 4 g .. 4 g + 11]
//          (K = 12 -> 16, a constant-1 input at k = 12 carries the bias in tap 0) with a banded weight image -- output n = d * 16 + c
//          (d = ow - 4 g) reads inputs k - d = 0..8 -- i.e. 5 row-shifted MMAs with N = 64 (32 for the last group): 15 MMAs instead of
//          one N = 16 GEMM per column (50), and a 13 KB window image instead of 42 KB.  The accumulators sit side by side in TMEM
//          columns 0..159 = ow * 16 + c, which is exactly conv2's K order (kw = ow, c) for the row: the epilogue (ReLU, fp16) writes
//          conv2's A image directly
//   conv2  2 row-shifted taps x 10 k-steps, N = 32 (columns 160..191); epilogue: bias, ReLU, AvgPool over row pairs (a lane shuffle)
//          -> conv3's A image (rows 0..11 of each window)
//   conv3  2 taps x 2 k-steps, N = 64 (columns 192..255); epilogue: bias, ReLU, AvgPool, the 320 -> 2 layer as per-lane partial dot
//          products + a warp sum, softplus, threshold
// One CTA = 128 threads and one tile at a time (thread 0 issues the copies and MMAs); two CTAs per SM (103 KB of shared memory, 256 TMEM
// columns each) overlap one tile's epilogues with the other's MMAs.  The sample's weight image (41 KB) stays in shared memory across tiles.
#pragma once

namespace cd3 {
constexpr int XQ_BYTES = 6 * CS;                    // window image of a tile: [3 column groups][2 chunks][132 rows][16 B]
constexpr int W1_BYTES = 5 * 2 * 64 * 16;           // [5 taps][2 chunks][64 n][16 B] (banded; the same image serves the three groups)
constexpr int W2_BYTES = 2 * 20 * 32 * 16;          // [2 taps][20 chunks][32 n][16 B]
constexpr int W3_BYTES = 2 * 4 * 64 * 16;           // [2 taps][4 chunks][64 n][16 B]
constexpr int L_W1 = 0, L_W2 = L_W1 + W1_BYTES, L_W3 = L_W2 + W2_BYTES, L_TAIL = L_W3 + W3_BYTES;
constexpr int T_B2 = 0, T_B3 = 32, T_W4 = 96, T_B4 = 96 + 640, TAIL_FLOATS = 96 + 640 + 2;  // fp32: b2[32] b3[64] W4[2][320] b4[2]
constexpr int IMG_BYTES = ((L_TAIL + TAIL_FLOATS * 4) + 255) / 256 * 256;
constexpr int IMG_HALVES = L_TAIL / 2;
// shared memory
constexpr int S_X = 0;                               // window image (+ 128 B zero slack: tap 4 reads two rows past the last chunk)
constexpr int S_A2 = S_X + XQ_BYTES + 128;           // conv2 A image: 20 chunks (k = ow * 16 + c)
constexpr int S_A3 = S_A2 + 20 * CS + 128;           // conv3 A image: 4 chunks
constexpr int S_W = S_A3 + 4 * CS + 128;             // weight image of the current sample
constexpr int S_BAR = S_W + IMG_BYTES;               // full @0, done @8, tmem slot @16
constexpr int SMEM = S_BAR + 64;
static_assert(SMEM <= 113 * 1024, "two Conv-D3 CTAs must fit one SM");
}  // namespace cd3

struct Cd3PackArgs {
  const float* w;
  long long w_stride;
  unsigned char* img;
  long long w_off[4], b_off[4];
};
// fp32 weights [S,P] -> per-sample fp16 images; thread = one image element
__global__ void tcc_pack_kernel(const Cd3PackArgs a) {
  const float* w = a.w + (long long)blockIdx.y * a.w_stride;
  unsigned char* img = a.img + (long long)blockIdx.y * cd3::IMG_BYTES;
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= cd3::IMG_HALVES + cd3::TAIL_FLOATS) return;
  if (e >= cd3::IMG_HALVES) {
    const int j = e - cd3::IMG_HALVES;
    float v;
    if (j < cd3::T_B3) v = w[a.b_off[1] + j];
    else if (j < cd3::T_W4) v = w[a.b_off[2] + j - cd3::T_B3];
    else if (j < cd3::T_B4) v = w[a.w_off[3] + j - cd3::T_W4];
    else v = w[a.b_off[3] + j - cd3::T_B4];
    *reinterpret_cast<float*>(img + cd3::L_TAIL + j * 4) = v;
    return;
  }
  float v = 0.f;
  if (e < cd3::L_W2 / 2) {  // conv1 [16,1,5,9], banded: (kh, chunk, n = d * 16 + c, j), k = chunk * 8 + j; kw = k - d; k == 12 of tap 0 = bias
    const int kh = e / 1024, r = e % 1024, ch = r / 512, n = (r % 512) >> 3, k = ch * 8 + (r & 7), d = n >> 4, c = n & 15, kw = k - d;
    if (k < 12 && kw >= 0 && kw < 9) v = w[a.w_off[0] + (c * 5 + kh) * 9 + kw];
    else if (k == 12 && kh == 0) v = w[a.b_off[0] + c];
  } else if (e < cd3::L_W3 / 2) {  // conv2 [32,16,2,10]: (kh, chunk cc, n, j), kw = cc / 2, c = (cc & 1) * 8 + j
    const int f = e - cd3::L_W2 / 2, kh = f / 5120, r = f % 5120, cc = r / 256, n = (r % 256) >> 3, c = (cc & 1) * 8 + (r & 7), kw = cc >> 1;
    v = w[a.w_off[1] + ((n * 16 + c) * 2 + kh) * 10 + kw];
  } else {  // conv3 [64,32,2,1]: (kh, chunk cc, n, j), c = cc * 8 + j
    const int f = e - cd3::L_W3 / 2, kh = f / 2048, r = f % 2048, cc = r / 512, n = (r % 512) >> 3, c = cc * 8 + (r & 7);
    v = w[a.w_off[2] + (n * 32 + c) * 2 + kh];
  }
  *reinterpret_cast<__half*>(img + 2 * e) = __float2half_rn(v);
}
// fp32 windows -> per-tile fp16 images [3 column groups][2 chunks][132 rows][16 B]: row (window q, time step t) of group g holds
// x[t][4 g + k], k = 0..11 (zero behind column 17), and a constant 1 at k = 12; thread = one 16-byte row of a chunk
__global__ void tcc_packx_kernel(const float* __restrict__ x, unsigned char* __restrict__ ximg, int B, int ntile) {
  const long long u = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (u >= (long long)ntile * 6 * ROWS) return;
  const int tile = (int)(u / (6 * ROWS)), v = (int)(u % (6 * ROWS)), ch = v / ROWS, r = v % ROWS;
  const int g = ch >> 1, c = ch & 1, rr = r - ROW0, q = rr >> 5, t = rr & 31, gw = tile * 4 + q;
  float f[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int k = c * 8 + j, col = 4 * g + k;
    f[j] = 0.f;
    if (rr >= 0 && rr < 128 && t < 30 && gw < B) f[j] = (k < 12 && col < 18) ? x[(long long)gw * 540 + t * 18 + col] : k == 12 ? 1.0f : 0.f;
  }
  *reinterpret_cast<uint4*>(ximg + (long long)tile * cd3::XQ_BYTES + ch * CS + r * 16) =
      make_uint4(pack_h2(f[0], f[1]), pack_h2(f[2], f[3]), pack_h2(f[4], f[5]), pack_h2(f[6], f[7]));
}

__device__ __forceinline__ void cd3_bulk(uint32_t dst, const unsigned char* src, int bytes, uint32_t bar) {
  for (int o = 0; o < bytes; o += 16384) bulk_g2s(dst + o, src + o, min(16384, bytes - o), bar);
}

struct Cd3Args {
  const unsigned char* ximg;  // [ntile][XQ_BYTES]
  const unsigned char* img;
  long long img_stride;
  int img_per, img_phase;  // MC sample s reads image (s + img_phase) / img_per
  float* out;  // [S,B,2]
  int B, S, ntile;
  int* status;
};

__global__ void __launch_bounds__(128, 2) tcc_kernel(const Cd3Args a) {
  using namespace cd3;
  extern __shared__ __align__(128) unsigned char smem[];
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t bar_full = sbase + S_BAR, bar_done = bar_full + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S_BAR + 16);
  // pad rows of the conv2 / conv3 A images, rows 12..31 of every window of conv3's, and the slack behind the window image stay zero
  for (int i = tid; i < (S_W - S_A2) / 16; i += 128) reinterpret_cast<uint4*>(smem + S_A2)[i] = make_uint4(0, 0, 0, 0);  // conv2 / conv3 A images
  for (int i = tid; i < 128 / 16; i += 128) reinterpret_cast<uint4*>(smem + S_X + XQ_BYTES)[i] = make_uint4(0, 0, 0, 0);
  if (tid == 0) {
    mbar_init(bar_full, 1);
    mbar_init(bar_done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), 256);
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t lane_base = tmem + ((uint32_t)(warp * 32) << 16);
  const float* tail = reinterpret_cast<const float*>(smem + S_W + L_TAIL);

  const long long total = (long long)a.S * a.ntile;
  const long long per = (total + gridDim.x - 1) / gridDim.x;
  const long long beg = per * blockIdx.x, end = min(total, beg + per);
  uint32_t fph = 0, dph = 0;
  int s_loaded = -1;
  bool ok = true, prefetched = false;
  const uint32_t xs = sbase + S_X, a2 = sbase + S_A2, a3 = sbase + S_A3, ws = sbase + S_W;

  auto layer_done = [&]() {
    ok = mbar_wait(bar_done, dph, a.status, 31) && ok;
    dph ^= 1u;
    tc_fence_after();
  };
  auto publish = [&]() {
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
  };

  for (long long it = beg; it < end && ok; ++it) {
    const int s = (int)(it / a.ntile), tile = (int)(it % a.ntile);
    if (tid == 0) {  // window image of the tile (+ the weight image when the MC sample changes), then conv1
      if (!prefetched) {
        const bool neww = s != s_loaded;
        mbar_expect_tx(bar_full, XQ_BYTES + (neww ? IMG_BYTES : 0));
        cd3_bulk(xs, a.ximg + (long long)tile * XQ_BYTES, XQ_BYTES, bar_full);
        if (neww) cd3_bulk(ws, a.img + (long long)((s + a.img_phase) / a.img_per) * a.img_stride, IMG_BYTES, bar_full);
      }
      ok = mbar_wait(bar_full, fph, a.status, 30) && ok;
      tc_fence_after();
#pragma unroll
      for (int g = 0; g < 3; ++g)
#pragma unroll
        for (int kh = 0; kh < 5; ++kh)
          umma(tmem + 64 * g, umma_desc(xs + 2 * g * CS + (ROW0 + kh) * 16, CS, 128), umma_desc(ws + L_W1 + kh * 2048, 1024, 128),
               g < 2 ? umma_idesc(64) : umma_idesc(32), kh != 0);
      umma_commit(bar_done);
    }
    s_loaded = s;
    fph ^= 1u;
    layer_done();
    // conv1's MMAs were the only readers of the window image: the next tile's travels underneath the rest of this tile (same MC sample
    // only: the weight image is still in use)
    prefetched = false;
    if (tid == 0 && it + 1 < end && (int)((it + 1) / a.ntile) == s) {
      mbar_expect_tx(bar_full, XQ_BYTES);
      cd3_bulk(xs, a.ximg + (long long)((it + 1) % a.ntile) * XQ_BYTES, XQ_BYTES, bar_full);
      prefetched = true;
    }
    const int q = warp, gw = tile * 4 + q;
    const uint32_t rowoff = (uint32_t)(ROW0 + tid) * 16;
    {  // conv1 epilogue: 10 x 16 channels -> ReLU -> conv2's A image (k = ow * 16 + c), rows >= 26 of a window are zero
      const bool live = lane < 26 && gw < a.B;
#pragma unroll 1
      for (int g0 = 0; g0 < 10; g0 += 5) {  // five 16-column loads in flight per wait
        float v[5][16];
#pragma unroll
        for (int g = 0; g < 5; ++g) tmem_ld16(lane_base + 16 * (g0 + g), v[g]);
        tmem_ld_wait();
#pragma unroll
        for (int g = 0; g < 5; ++g) {
          uint4 lo = make_uint4(0, 0, 0, 0), hi = lo;
          if (live) {
            lo = make_uint4(pack_relu_h2(v[g][0], v[g][1]), pack_relu_h2(v[g][2], v[g][3]), pack_relu_h2(v[g][4], v[g][5]), pack_relu_h2(v[g][6], v[g][7]));
            hi = make_uint4(pack_relu_h2(v[g][8], v[g][9]), pack_relu_h2(v[g][10], v[g][11]), pack_relu_h2(v[g][12], v[g][13]), pack_relu_h2(v[g][14], v[g][15]));
          }
          *reinterpret_cast<uint4*>(smem + S_A2 + (2 * (g0 + g)) * CS + rowoff) = lo;
          *reinterpret_cast<uint4*>(smem + S_A2 + (2 * (g0 + g) + 1) * CS + rowoff) = hi;
        }
      }
    }
    publish();
    if (tid == 0) {
      tc_fence_after();
#pragma unroll
      for (int kh = 0; kh < 2; ++kh)
        for (int ks = 0; ks < 10; ++ks)
          umma(tmem + 160, umma_desc(a2 + 2 * ks * CS + (ROW0 + kh) * 16, CS, 128), umma_desc(ws + L_W2 + kh * 10240 + 2 * ks * 512, 512, 128),
               umma_idesc(32), (kh | ks) != 0);
      umma_commit(bar_done);
    }
    layer_done();
    {  // conv2 epilogue: bias, ReLU, AvgPool((2,1)) over rows (2 j, 2 j + 1), j < 12 -> conv3's A image row j of the window
      float v[2][16];
      tmem_ld16(lane_base + 160, v[0]);
      tmem_ld16(lane_base + 176, v[1]);
      tmem_ld_wait();
      uint32_t h[16];
#pragma unroll
      for (int c = 0; c < 32; c += 2) {
        float p0 = fmaxf(v[c >> 4][c & 15] + tail[T_B2 + c], 0.f), p1 = fmaxf(v[c >> 4][(c & 15) + 1] + tail[T_B2 + c + 1], 0.f);
        p0 = 0.5f * (p0 + __shfl_down_sync(0xffffffffu, p0, 1));
        p1 = 0.5f * (p1 + __shfl_down_sync(0xffffffffu, p1, 1));
        h[c >> 1] = pack_h2(p0, p1);
      }
      if (!(lane & 1) && lane < 24) {
        const bool live = gw < a.B;
        unsigned char* dst = smem + S_A3 + (ROW0 + q * 32 + (lane >> 1)) * 16;
#pragma unroll
        for (int cc = 0; cc < 4; ++cc)
          *reinterpret_cast<uint4*>(dst + cc * CS) = live ? make_uint4(h[4 * cc], h[4 * cc + 1], h[4 * cc + 2], h[4 * cc + 3]) : make_uint4(0, 0, 0, 0);
      }
    }
    publish();
    if (tid == 0) {
      tc_fence_after();
#pragma unroll
      for (int kh = 0; kh < 2; ++kh)
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
          umma(tmem + 192, umma_desc(a3 + 2 * ks * CS + (ROW0 + kh) * 16, CS, 128), umma_desc(ws + L_W3 + kh * 4096 + 2 * ks * 1024, 1024, 128),
               umma_idesc(64), (kh | ks) != 0);
      umma_commit(bar_done);
    }
    layer_done();
    {  // conv3 epilogue: bias, ReLU, AvgPool over rows (2 j, 2 j + 1), j < 5; Linear(320, 2) over (c, j) = c * 5 + j; softplus; threshold
      float o0 = 0.f, o1 = 0.f;
      const int j = lane >> 1;
      const bool mine = !(lane & 1) && lane < 10;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float v[16];
        tmem_ld16(lane_base + 192 + 16 * g, v);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int c = g * 16 + i;
          float p = fmaxf(v[i] + tail[T_B3 + c], 0.f);
          p = 0.5f * (p + __shfl_down_sync(0xffffffffu, p, 1));
          if (mine) {
            o0 = fmaf(p, tail[T_W4 + c * 5 + j], o0);
            o1 = fmaf(p, tail[T_W4 + 320 + c * 5 + j], o1);
          }
        }
      }
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) {
        o0 += __shfl_xor_sync(0xffffffffu, o0, d);
        o1 += __shfl_xor_sync(0xffffffffu, o1, d);
      }
      if (lane == 0 && gw < a.B) {
        o0 += tail[T_B4];
        o1 += tail[T_B4 + 1];
        o0 = o0 > 20.f ? o0 : log1pf(expf(o0));
        o1 = o1 > 20.f ? o1 : log1pf(expf(o1));
        *reinterpret_cast<float2*>(a.out + ((long long)s * a.B + gw) * 2) = make_float2(o0 > 1e-9f ? o0 : 1e-9f, o1 > 1e-9f ? o1 : 1e-9f);
      }
    }
    tc_fence_before();
    __syncthreads();  // accumulators drained before the next tile's MMAs overwrite them
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 256);
}
