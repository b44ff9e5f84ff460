// tcgen05 predictive engine for the Linear net (nets/linear.py:44-55, 66-70: flatten 540 -> 256 -> 128 -> 128 -> 32 -> 2, ReLU between the
// layers, softplus + Threshold(1e-9) on both outputs); DET / weight-sampling forward without dropout.  Included by brl_tc.cu.
//
// One persistent CTA per SM, 128 threads (thread = window of a 128-window tile = TMEM lane).  Per (MC sample, window tile):
//   fc1  A = the windows as an fp16 matrix [B padded to 128][576] (540 inputs + zero padding), 128 x 64 boxes through a TMA tensor map
//        (SWIZZLE_128B); B = the sample's fp16 weight image, k-blocks of 64 inputs x 256 outputs (32 KB, UMMA canonical K-major),
//        bulk-copied; both through a two-stage shared-memory ring; accumulator = TMEM columns 0..255
//   fc2..fc4  A = the previous layer's activations, written by the epilogue as fp16 K-major chunks [8 inputs][128 windows][16 B] in
//        shared memory (never in HBM); B streamed through the ring; accumulators = TMEM columns 256..383, 384..511, 0..31
//   head 32 -> 2, softplus and the threshold in registers.
// Thread 0 issues every copy and MMA of a layer and commits to `done`; all threads run the epilogue.  A tile-sample moves 395 KB of
// weights + 144 KB of windows out of L2 for 49 MFLOP, so the kernel is bound by that feed, not by the tensor pipe.
#pragma once

namespace lin {
constexpr int KX = 576;                       // fc1 K padded to 9 k-blocks of 64
constexpr int NKB1 = KX / 64;
constexpr int N1 = 256, N2 = 128, N3 = 128, N4 = 32;
constexpr int KB1_BYTES = 8 * N1 * 16, KB2_BYTES = 8 * N2 * 16, KB3_BYTES = 8 * N3 * 16, KB4_BYTES = 8 * N4 * 16;
constexpr int L_W1 = 0, L_W2 = L_W1 + NKB1 * KB1_BYTES, L_W3 = L_W2 + 4 * KB2_BYTES, L_W4 = L_W3 + 2 * KB3_BYTES;
constexpr int L_TAIL = L_W4 + 2 * KB4_BYTES;  // fp32: b1[256] b2[128] b3[128] b4[32] W5[2][32] b5[2]
constexpr int T_B1 = 0, T_B2 = 256, T_B3 = 384, T_B4 = 512, T_W5 = 544, T_B5 = 608, TAIL_FLOATS = 610;
constexpr int IMG_BYTES = ((L_TAIL + TAIL_FLOATS * 4) + 255) / 256 * 256;
constexpr int IMG_HALVES = L_TAIL / 2;
// shared memory
constexpr int STAGE_A = 128 * 128;            // one TMA box: 128 windows x 64 fp16
constexpr int STAGE_BYTES = STAGE_A + KB1_BYTES;
constexpr int S_H1 = 2 * STAGE_BYTES;         // 32 chunks x 2 KB
constexpr int S_H2 = S_H1 + 32 * 2048;        // 16 chunks; h3 aliases h1
constexpr int S_BAR = S_H2 + 16 * 2048;       // full[2] @0, empty[2] @16, done @32, tmem slot @40
constexpr int SMEM = S_BAR + 64 + 1024;       // + slack to align the ring to 1024 B (SWIZZLE_128B atoms)
static_assert(SMEM <= 232448, "linear kernel shared memory exceeds the opt-in limit");
}  // namespace lin

struct LinPackArgs {
  const float* w;
  long long w_stride;  // P, or 0 when the weights are shared by all samples
  unsigned char* img;
  long long w_off[5], b_off[5];
};
// fp32 weights [S,P] -> per-sample fp16 images; thread = one image element
__global__ void tcl_pack_kernel(const LinPackArgs a) {
  const int s = blockIdx.y;
  const float* w = a.w + (long long)s * a.w_stride;
  unsigned char* img = a.img + (long long)s * lin::IMG_BYTES;
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= lin::IMG_HALVES + lin::TAIL_FLOATS) return;
  if (e >= lin::IMG_HALVES) {
    const int j = e - lin::IMG_HALVES;
    float v;
    if (j < lin::T_B2) v = w[a.b_off[0] + j];
    else if (j < lin::T_B3) v = w[a.b_off[1] + j - lin::T_B2];
    else if (j < lin::T_B4) v = w[a.b_off[2] + j - lin::T_B3];
    else if (j < lin::T_W5) v = w[a.b_off[3] + j - lin::T_B4];
    else if (j < lin::T_B5) v = w[a.w_off[4] + j - lin::T_W5];
    else v = w[a.b_off[4] + j - lin::T_B5];
    *reinterpret_cast<float*>(img + lin::L_TAIL + j * 4) = v;
    return;
  }
  int layer, N, K;
  if (e < lin::L_W2 / 2) { layer = 0; N = lin::N1; K = 540; }
  else if (e < lin::L_W3 / 2) { layer = 1; N = lin::N2; K = 256; e -= lin::L_W2 / 2; }
  else if (e < lin::L_W4 / 2) { layer = 2; N = lin::N3; K = 128; e -= lin::L_W3 / 2; }
  else { layer = 3; N = lin::N4; K = 128; e -= lin::L_W4 / 2; }
  // k-block [8 chunks][N][8]: element (kb, c, n, j) is input k = kb * 64 + c * 8 + j of output n
  const int per_kb = 64 * N, kb = e / per_kb, r = e - kb * per_kb, c = r / (8 * N), r2 = r - c * 8 * N, n = r2 >> 3, j = r2 & 7;
  const int k = kb * 64 + c * 8 + j;
  const float v = k < K ? w[a.w_off[layer] + (long long)n * K + k] : 0.f;
  const int base = layer == 0 ? lin::L_W1 : layer == 1 ? lin::L_W2 : layer == 2 ? lin::L_W3 : lin::L_W4;
  *reinterpret_cast<__half*>(img + base + 2 * (kb * per_kb + r)) = __float2half_rn(v);
}
// fp32 windows [B,540] -> fp16 matrix [Bpad][576] (zero rows / columns behind B / 540); thread = 8 columns of a row
__global__ void tcl_packx_kernel(const float* __restrict__ x, unsigned char* __restrict__ x16, int B, int Bpad) {
  const long long u = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (u >= (long long)Bpad * (lin::KX / 8)) return;
  const int row = (int)(u / (lin::KX / 8)), g = (int)(u % (lin::KX / 8));
  float f[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int k = g * 8 + j;
    f[j] = (row < B && k < 540) ? x[(long long)row * 540 + k] : 0.f;
  }
  *reinterpret_cast<uint4*>(x16 + ((long long)row * lin::KX + g * 8) * 2) =
      make_uint4(pack_h2(f[0], f[1]), pack_h2(f[2], f[3]), pack_h2(f[4], f[5]), pack_h2(f[6], f[7]));
}

struct LinArgs {
  const unsigned char* img;
  long long img_stride;  // IMG_BYTES or 0
  int img_per, img_phase;  // MC sample s reads image (s + img_phase) / img_per
  float* out;            // [S,B,2]
  int B, S, ntile128;
  int* status;
};

__global__ void __launch_bounds__(128, 1) tcl_kernel(const LinArgs a, const __grid_constant__ CUtensorMap xmap) {
  using namespace lin;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t bars = sbase + S_BAR;
  const uint32_t bar_full = bars, bar_empty = bars + 16, bar_done = bars + 32;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S_BAR + 40);
  if (tid == 0) {
    for (int i = 0; i < 2; ++i) { mbar_init(bar_full + 8 * i, 1); mbar_init(bar_empty + 8 * i, 1); }
    mbar_init(bar_done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t lane_base = tmem + ((uint32_t)(warp * 32) << 16);

  const long long total = (long long)a.S * a.ntile128;
  const long long per = (total + gridDim.x - 1) / gridDim.x;
  const long long beg = per * blockIdx.x, end = min(total, beg + per);
  uint32_t ld_cnt = 0, use_cnt = 0, dph = 0;  // ring counters (thread 0) and the parity of `done` (all threads)
  bool ok = true;

  for (long long it = beg; it < end && ok; ++it) {
    const int s = (int)(it / a.ntile128), tile = (int)(it % a.ntile128);
    const unsigned char* img = a.img + (long long)((s + a.img_phase) / a.img_per) * a.img_stride;
    const float* tail = reinterpret_cast<const float*>(img + L_TAIL);
    const int row0 = tile * 128;

    // one layer's copies and MMAs (thread 0): k-blocks of 64 through the two-stage ring, the first two copies may already be in flight
    auto load = [&](bool tma_a, int kb, const unsigned char* wsrc, int wbytes, int xrow = -1) {
      const uint32_t st = ld_cnt & 1u;
      if (ld_cnt >= 2) ok = mbar_wait(bar_empty + 8 * st, ((ld_cnt - 2) >> 1) & 1u, a.status, 20) && ok;  // the MMAs that read the stage
      const uint32_t dst = sbase + st * STAGE_BYTES;
      mbar_expect_tx(bar_full + 8 * st, (tma_a ? STAGE_A : 0) + wbytes);
      if (tma_a) tma_load_2d(dst, &xmap, kb * 64, xrow >= 0 ? xrow : row0, bar_full + 8 * st);
      bulk_g2s(dst + STAGE_A, wsrc + (long long)kb * wbytes, wbytes, bar_full + 8 * st);
      ++ld_cnt;
    };
    auto run_layer = [&](bool tma_a, int nkb, uint32_t a_smem, int N, const unsigned char* wsrc, int wbytes, uint32_t tcol, int preloaded) {
      for (int kb = preloaded; kb < min(2, nkb); ++kb) load(tma_a, kb, wsrc, wbytes);
      for (int kb = 0; kb < nkb && ok; ++kb) {
        const uint32_t st = use_cnt & 1u;
        ok = mbar_wait(bar_full + 8 * st, (use_cnt >> 1) & 1u, a.status, 21) && ok;
        tc_fence_after();
        const uint32_t sa = sbase + st * STAGE_BYTES, sb = sa + STAGE_A;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          const uint64_t da = tma_a ? umma_desc_sw128(sa + ks * 32) : umma_desc(a_smem + (uint32_t)(kb * 8 + 2 * ks) * 2048u, 2048, 128);
          umma(tmem + tcol, da, umma_desc(sb + 2 * ks * (N * 16), N * 16, 128), umma_idesc(N), (kb | ks) != 0);
        }
        umma_commit(bar_empty + 8 * st);
        ++use_cnt;
        if (kb + 2 < nkb) load(tma_a, kb + 2, wsrc, wbytes);
      }
      umma_commit(bar_done);
    };
    // epilogue: NCOL accumulator columns of this thread's window -> bias, ReLU, fp16 K-major chunks at `dst` (chunk stride 2 KB)
    auto store_act = [&](uint32_t tcol, int ncol, const float* bias, unsigned char* dst) {
      for (int g = 0; g < ncol / 16; ++g) {
        float v[16];
        tmem_ld16(lane_base + tcol + g * 16, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j] + __ldg(bias + g * 16 + j), 0.f);
        unsigned char* p = dst + (2 * g) * 2048 + tid * 16;
        *reinterpret_cast<uint4*>(p) = make_uint4(pack_h2(v[0], v[1]), pack_h2(v[2], v[3]), pack_h2(v[4], v[5]), pack_h2(v[6], v[7]));
        *reinterpret_cast<uint4*>(p + 2048) = make_uint4(pack_h2(v[8], v[9]), pack_h2(v[10], v[11]), pack_h2(v[12], v[13]), pack_h2(v[14], v[15]));
      }
    };
    auto layer_done = [&]() {
      ok = mbar_wait(bar_done, dph, a.status, 22) && ok;
      dph ^= 1u;
      tc_fence_after();
    };
    auto publish = [&]() {  // activations written: visible to the MMAs (async proxy) of the next layer
      fence_async_smem();
      tc_fence_before();
      __syncthreads();
    };

    if (tid == 0) run_layer(true, NKB1, 0u, N1, img + L_W1, KB1_BYTES, 0u, it == beg ? 0 : 2);  // (first two copies: end of the previous item)
    layer_done();
    if (tid == 0) { load(false, 0, img + L_W2, KB2_BYTES); load(false, 1, img + L_W2, KB2_BYTES); }  // underneath the epilogue
    store_act(0u, N1, tail + T_B1, smem + S_H1);
    publish();
    if (tid == 0) { tc_fence_after(); run_layer(false, 4, sbase + S_H1, N2, img + L_W2, KB2_BYTES, 256u, 2); }
    layer_done();
    if (tid == 0) { load(false, 0, img + L_W3, KB3_BYTES); load(false, 1, img + L_W3, KB3_BYTES); }
    store_act(256u, N2, tail + T_B2, smem + S_H2);
    publish();
    if (tid == 0) { tc_fence_after(); run_layer(false, 2, sbase + S_H2, N3, img + L_W3, KB3_BYTES, 384u, 2); }
    layer_done();
    if (tid == 0) { load(false, 0, img + L_W4, KB4_BYTES); load(false, 1, img + L_W4, KB4_BYTES); }
    store_act(384u, N3, tail + T_B3, smem + S_H1);  // h3 aliases h1 (its readers, the fc2 MMAs, completed before fc3 was issued)
    publish();
    if (tid == 0) { tc_fence_after(); run_layer(false, 2, sbase + S_H1, N4, img + L_W4, KB4_BYTES, 0u, 2); }
    layer_done();
    if (tid == 0 && it + 1 < end) {  // the ring is idle from here on: the next item's first two fc1 k-blocks travel underneath the head
      const int s2 = (int)((it + 1) / a.ntile128), tile2 = (int)((it + 1) % a.ntile128);
      const unsigned char* img2 = a.img + (long long)((s2 + a.img_phase) / a.img_per) * a.img_stride;
      load(true, 0, img2 + L_W1, KB1_BYTES, tile2 * 128);
      load(true, 1, img2 + L_W1, KB1_BYTES, tile2 * 128);
    }
    // fc4 epilogue + head 32 -> 2 + softplus + Threshold(1e-9, 1e-9)
    {
      float o0 = __ldg(tail + T_B5), o1 = __ldg(tail + T_B5 + 1);
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        float v[16];
        tmem_ld16(lane_base + g * 16, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float h = fmaxf(v[j] + __ldg(tail + T_B4 + g * 16 + j), 0.f);
          o0 = fmaf(h, __ldg(tail + T_W5 + g * 16 + j), o0);
          o1 = fmaf(h, __ldg(tail + T_W5 + 32 + g * 16 + j), o1);
        }
      }
      const int gw = row0 + tid;
      if (gw < a.B) {
        o0 = o0 > 20.f ? o0 : log1pf(expf(o0));
        o1 = o1 > 20.f ? o1 : log1pf(expf(o1));
        *reinterpret_cast<float2*>(a.out + ((long long)s * a.B + gw) * 2) = make_float2(o0 > 1e-9f ? o0 : 1e-9f, o1 > 1e-9f ? o1 : 1e-9f);
      }
    }
    tc_fence_before();
    __syncthreads();  // every accumulator column is drained before the next tile's fc1 overwrites columns 0..255
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512);
}
