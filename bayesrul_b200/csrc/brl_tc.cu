// tcgen05 / TMEM engine for the Inception regressor (fp16 operands, fp32 accumulation in TMEM).
//
// Three kernels per chunk of MC samples:
//   tc_pack_kernel  fp32 weight draws [S,P] -> per-sample fp16 images in the UMMA canonical K-major
//                   (no-swizzle) layout, i.e. exactly the bytes the MMA descriptors address
//   tc_conv_kernel  persistent, one CTA per SM: the whole conv stack (both inception modules) of a
//                   128-row tile (4 windows x 32 rows) stays in SMEM/TMEM; weights of the current MC
//                   sample are staged once per sample by cp.async.bulk (1-D TMA) and stay resident;
//                   'same' padding = shifted A descriptors over zero pad rows; epilogues (bias, ReLU,
//                   dropout, fp16 pack, max-pool) run TMEM -> registers -> SMEM (next layer's A operand)
//   tc_fc_kernel    warp-specialised GEMM [128 windows x 2400] x [2400 x 64] per (sample, window tile):
//                   bulk-copy producer warp / single-thread tcgen05.mma issuer / 4 epilogue warps with a
//                   double-buffered TMEM accumulator; epilogue fuses bias, ReLU, dropout, the 64->2
//                   head, softplus and Threshold(1e-9).
// Reference semantics: nets/inception.py:54-61,125-132,211-215 (SURVEY Appendix B).
#include <cuda_fp16.h>

#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <utility>
#include <vector>

#include <cuda.h>

#include "../../include/bayesrul_b200.h"
#include "brl_kernels.cuh"
#include "brl_nets.h"
#include "brl_philox.cuh"
#include "brl_tc.cuh"
#include "brl_tc_ptx.cuh"

namespace brl {

// ------------------------------------------------------------------------------------------------
// geometry
// ------------------------------------------------------------------------------------------------
constexpr int ROWS = 132;            // 2 zero rows + 128 tile rows + 2 slack rows
constexpr int CS = ROWS * 16;        // bytes of one 8-channel chunk (K-major, 16 B per row)
constexpr int ROW0 = 2;              // buffer row of tile row 0
// per-slot activation region: 32 chunks; M1 | M1P, with T2/T3 aliasing M1 and X/XP aliasing M1P
constexpr int R_M1 = 0;                     // 16 chunks: 4 branches x (27 real + const-1 + zero pad = 32)
constexpr int R_M1P = 16 * CS;              // 16 chunks
constexpr int R_T2 = R_M1, R_T3 = R_M1 + 8 * CS;   // 8 + 8 chunks (live after the M1 readers have completed)
constexpr int R_X = R_M1P, R_XP = R_M1P + 3 * CS;  // 3 + 3 chunks (live before M1P is produced), one bulk copy
constexpr int G_BYTES = 32 * CS;
constexpr int OFF_W = 2 * G_BYTES;          // weight image, shared by the two groups
// weight image (identical in the global blob)
constexpr int WA_TAP = 4 * 32 * 16;         // [4 chunks][32 n][16 B]
constexpr int WI_A = 0;                     // 12 taps
constexpr int WI_B1 = WI_A + 12 * WA_TAP;   // [16 chunks][144 n][16 B]
constexpr int WI_B4 = WI_B1 + 16 * 144 * 16;  // [16 chunks][32 n][16 B]
constexpr int WC_TAP = 8 * 16 * 16;         // [8 chunks][16 n][16 B]
constexpr int WI_B2B = WI_B4 + 16 * 32 * 16;  // 3 taps
constexpr int WI_B3B = WI_B2B + 3 * WC_TAP;   // 5 taps
constexpr int WI_BIAS = WI_B3B + 5 * WC_TAP;  // fp32: A 4x32, B1 144, B4 32, b2b 16, b3b 16
constexpr int NBIAS = 128 + 144 + 32 + 16 + 16;
constexpr int CONV_IMG = WI_BIAS + NBIAS * 4;
static_assert(CONV_IMG % 16 == 0, "bulk copies need 16-byte multiples");
constexpr int OFF_ZERO = OFF_W + CONV_IMG;    // one all-zero chunk: the 4th K chunk of X / XP of both slots
constexpr int OFF_BAR = OFF_ZERO + CS;
constexpr int CONV_SMEM = OFF_BAR + 256;
constexpr int XIMG_TILE_BYTES = 6 * CS;       // fp16 chunk images of a tile's windows: X0 X1 X2 XP0 XP1 XP2, pad rows included
static_assert(CONV_SMEM <= 232448, "conv kernel shared memory exceeds the 227 KB opt-in limit");
// blob = conv image + fc image + fp32 tail (fc bias 64, last W 128, last b 2)
constexpr int FC_KPAD = 2432;                // K of the fc GEMM padded to 38 x 64 (zero weights behind 2400)
constexpr int FC_IMG = (FC_KPAD / 8) * 64 * 16;  // [304 k-chunks][64 n][16 B]
constexpr int BLOB_FC = CONV_IMG;
constexpr int BLOB_TAIL = BLOB_FC + FC_IMG;
constexpr int BLOB_BYTES = ((BLOB_TAIL + 194 * 4) + 255) / 256 * 256;
constexpr int FEAT_ROW_BYTES = 4800;         // feature tensor: row-major [S][Bpad][2400] fp16, k' = (c / 8) * 240 + t * 8 + c % 8
// fc kernel: A = 128 windows x 64 k per stage through a TMA tensor map (SWIZZLE_128B), B = 8 k-chunks of the weight image
constexpr int FC_BK = 64;
constexpr int FC_NKB = FC_KPAD / FC_BK;      // 38 (the last box is half out of bounds: TMA fills zeros)
constexpr int FC_STAGES = 6;
constexpr int FC_A_BYTES = 128 * 128, FC_W_BYTES = (FC_BK / 8) * 1024;
constexpr int FC_STAGE_BYTES = FC_A_BYTES + FC_W_BYTES;
constexpr int FC_SMEM = FC_STAGES * FC_STAGE_BYTES + 256 + 1024;  // + barriers + slack to align the ring to 1024 B

struct TcState {
  int net;
  int* status;  // device: 0 ok, else first mbarrier time-out code
  int sm_count;
  long long loff[12][2];  // w_off, b_off per layer
  bool timing = false;    // bracket tc_conv_kernel launches with events (bench.py roofline)
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> evs[2];  // 0: tc_conv_kernel, 1: tc_fc_kernel
  size_t ev_used[2] = {0, 0};
  long long* trace = nullptr;
};

// ------------------------------------------------------------------------------------------------
// weight packing: fp32 [S,P] -> fp16 images
// ------------------------------------------------------------------------------------------------
struct PackArgs {
  const float* w;
  long long w_stride;  // P, or 0 when the weights are shared by all samples
  unsigned char* blob;
  long long off[12][2];
  // inverted dropout's 1 / keep of the sites behind module 1 and module 2 (MC-dropout: 1 / (1 - p / 4), else 1), folded into the
  // weights that read those activations: the module-2 1x1 convs and the fc layer (their bias entries are not scaled)
  float inv4;
};

__device__ __forceinline__ void put_h(unsigned char* img, int byte_off, float v) {
  *reinterpret_cast<__half*>(img + byte_off) = __float2half_rn(v);
}

__global__ void tc_pack_kernel(const PackArgs a) {
  const int s = blockIdx.y;
  const float* w = a.w + (long long)s * a.w_stride;
  unsigned char* blob = a.blob + (long long)s * BLOB_BYTES;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  constexpr int N_A = 12 * 32 * 32, N_B1 = 144 * 128, N_B4 = 32 * 128, N_C2 = 3 * 16 * 64, N_C3 = 5 * 16 * 64;
  constexpr int N_FC = 64 * FC_KPAD;
  int j = i;
  if (j < N_A) {  // module 1: tap-major [tap][k/8][n][k%8]
    const int tap = j / 1024, r = j % 1024, n = r / 32, k = r % 32;
    const int layer = tap == 0 ? 0 : tap < 4 ? 1 : tap < 9 ? 2 : 3;
    const int t0 = layer == 0 ? 0 : layer == 1 ? 1 : layer == 2 ? 4 : 9;
    const int ntap = layer == 0 ? 1 : layer == 2 ? 5 : 3;
    const int tl = tap - t0, padl = ntap >> 1;
    float v = 0.f;
    if (n < 27 && k < 18) v = w[a.off[layer][0] + ((long long)n * 18 + k) * ntap + tl];
    else if (k == 18 && tl == padl && n < 27) v = w[a.off[layer][1] + n];  // bias rides on the constant-1 feature
    else if (k == 18 && layer == 0 && n == 27) v = 1.0f;                  // conv1 column 27 re-emits the constant into M1
    int dst;
    if (layer == 3) {  // pooled branch: one [4 chunks][32][16 B] tile per tap
      dst = WI_A + 18432 + tl * 2048 + (k >> 3) * 512 + n * 16 + (k & 7) * 2;
    } else {           // x branches: one tile per input shift, rows = conv5 | conv3 | conv1
      const int sh = tl - padl;
      const int q = sh == 0 ? 0 : sh == -1 ? 1 : sh == 1 ? 2 : sh == -2 ? 3 : 4;
      const int nsh = q == 0 ? 96 : q < 3 ? 64 : 32;
      const int osh = q == 0 ? 0 : q == 1 ? 6144 : q == 2 ? 10240 : q == 3 ? 14336 : 16384;
      const int nrow = (layer == 2 ? 0 : layer == 1 ? 32 : 64) + n;
      dst = WI_A + osh + (k >> 3) * (nsh * 16) + nrow * 16 + (k & 7) * 2;
    }
    put_h(blob, dst, v);
    return;
  }
  j -= N_A;
  if (j < N_B1) {  // module-2 1x1 convs of b1 | b2a | b3a over the padded M1 channels
    const int n = j / 128, k = j % 128;
    const int layer = n < 16 ? 4 : n < 80 ? 5 : 7;
    const int co = n < 16 ? n : n < 80 ? n - 16 : n - 80;
    const int grp = k >> 5, c = k & 31;
    float v = 0.f;
    if (c < 27) v = a.inv4 * w[a.off[layer][0] + (long long)co * 108 + grp * 27 + c];
    else if (k == 27) v = w[a.off[layer][1] + co];  // bias on M1's constant channel
    put_h(blob, WI_B1 + (k >> 3) * (144 * 16) + n * 16 + (k & 7) * 2, v);
    return;
  }
  j -= N_B1;
  if (j < N_B4) {
    const int n = j / 128, k = j % 128, grp = k >> 5, c = k & 31;
    float v = 0.f;
    if (c < 27) v = a.inv4 * w[a.off[9][0] + (long long)n * 108 + grp * 27 + c];
    else if (k == 27) v = w[a.off[9][1] + n];
    put_h(blob, WI_B4 + (k >> 3) * 512 + n * 16 + (k & 7) * 2, v);
    return;
  }
  j -= N_B4;
  if (j < N_C2) {
    const int tap = j / 1024, r = j % 1024, n = r / 64, k = r % 64;
    put_h(blob, WI_B2B + (k >> 3) * 768 + (tap * 16 + n) * 16 + (k & 7) * 2, w[a.off[6][0] + ((long long)n * 64 + k) * 3 + tap]);
    return;
  }
  j -= N_C2;
  if (j < N_C3) {
    const int tap = j / 1024, r = j % 1024, n = r / 64, k = r % 64;
    put_h(blob, WI_B3B + (k >> 3) * 1280 + (tap * 16 + n) * 16 + (k & 7) * 2, w[a.off[8][0] + ((long long)n * 64 + k) * 5 + tap]);
    return;
  }
  j -= N_C3;
  if (j < NBIAS) {
    float v = 0.f;
    if (j < 128) { const int br = j >> 5, c = j & 31; if (c < 27) v = w[a.off[br][1] + c]; }
    else if (j < 272) { const int n = j - 128; v = n < 16 ? w[a.off[4][1] + n] : n < 80 ? w[a.off[5][1] + n - 16] : w[a.off[7][1] + n - 80]; }
    else if (j < 304) v = w[a.off[9][1] + j - 272];
    else if (j < 320) v = w[a.off[6][1] + j - 304];
    else v = w[a.off[8][1] + j - 320];
    *reinterpret_cast<float*>(blob + WI_BIAS + j * 4) = v;
    return;
  }
  j -= NBIAS;
  if (j < N_FC) {  // fc: k' = (c / 8) * 240 + t * 8 + c % 8  <-  original column c*30 + t; zero behind 2400
    const int n = j / FC_KPAD, kp = j % FC_KPAD;
    float v = 0.f;
    if (kp < 2400) {
      const int cb = kp / 240, r = kp % 240, t = r >> 3, c = cb * 8 + (r & 7);
      v = a.inv4 * w[a.off[10][0] + (long long)n * 2400 + c * 30 + t];
    }
    put_h(blob, BLOB_FC + (kp >> 3) * 1024 + n * 16 + (kp & 7) * 2, v);
    return;
  }
  j -= N_FC;
  if (j < 194) {
    float v = j < 64 ? w[a.off[10][1] + j] : j < 192 ? w[a.off[11][0] + j - 64] : w[a.off[11][1] + j - 192];
    *reinterpret_cast<float*>(blob + BLOB_TAIL + j * 4) = v;
  }
}
constexpr int PACK_THREADS_TOTAL = 12 * 1024 + 144 * 128 + 32 * 128 + 3 * 1024 + 5 * 1024 + NBIAS + 64 * FC_KPAD + 194;

#include "brl_tc_conv.cuh"

// ------------------------------------------------------------------------------------------------
// fc + head kernel
// ------------------------------------------------------------------------------------------------
struct FcArgs {
  const unsigned char* blob;
  long long blob_stride;
  int img_per, img_phase;  // MC sample s reads image (s + img_phase) / img_per (ConvArgs)
  float* out;  // [S,B,2]
  int B, S, ntile128;  // feature rows per sample = ntile128 * 128
  float keep;  // dropout keep of the fc site
  NoiseRef drop;
  int* status;
};

// K-major SWIZZLE_128B shared-memory matrix descriptor (what a TMA SWIZZLE_128B box of 64 fp16 columns produces):
// 8-row x 128-byte atoms of 1024 B, SBO = 1024 between 8-row groups, layout type 2; k advances by +32 B inside the atom
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | (1ull << 16) | ((uint64_t)(1024u >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar)
      : "memory");
}

template <bool DROP>
__global__ void __launch_bounds__(192, 1) tc_fc_kernel(const FcArgs a, const __grid_constant__ CUtensorMap fmap) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // SWIZZLE_128B atoms: 1024-byte aligned
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t bars = sbase + FC_STAGES * FC_STAGE_BYTES;
  // full[6] @0, empty[6] @48, tmem_full[2] @96, tmem_empty[2] @112, tmem slot @128
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + FC_STAGES * FC_STAGE_BYTES + 128);
  if (tid == 0) {
    for (int i = 0; i < FC_STAGES; ++i) { mbar_init(bars + 8 * i, 1); mbar_init(bars + 48 + 8 * i, 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(bars + 96 + 8 * i, 1); mbar_init(bars + 112 + 8 * i, 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), 128);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const long long total = (long long)a.S * a.ntile128;
  constexpr int NKB = FC_NKB;

  if (warp == 0) {
    if (lane == 0) {  // ===== producer: bulk copies of the A (features) and B (fc weights) k-blocks
      uint32_t stage = 0, ph = 1;
      bool ok = true;
      for (long long it = blockIdx.x; it < total && ok; it += gridDim.x) {
        const int s = (int)(it / a.ntile128);
        const int row0 = (int)(it * 128);  // == (s * ntile128 + tile) * 128: rows of the [S * Bpad, 2400] feature matrix
        const unsigned char* gb = a.blob + (long long)((s + a.img_phase) / a.img_per) * a.blob_stride + BLOB_FC;
        for (int kb = 0; kb < NKB && ok; ++kb) {
          ok = mbar_wait(bars + 48 + 8 * stage, ph, a.status, 10);
          const uint32_t dst = sbase + stage * FC_STAGE_BYTES;
          mbar_expect_tx(bars + 8 * stage, FC_STAGE_BYTES);
          tma_load_2d(dst, &fmap, kb * FC_BK, row0, bars + 8 * stage);
          bulk_g2s(dst + FC_A_BYTES, gb + (long long)kb * FC_W_BYTES, FC_W_BYTES, bars + 8 * stage);
          if (++stage == FC_STAGES) { stage = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {  // ===== single-thread MMA issuer
      constexpr uint32_t idesc = umma_idesc(64);
      uint32_t stage = 0, ph = 0, acc_i = 0, aph = 1;
      bool ok = true;
      for (long long it = blockIdx.x; it < total && ok; it += gridDim.x) {
        ok = mbar_wait(bars + 112 + 8 * acc_i, aph, a.status, 11);
        tc_fence_after();
        for (int kb = 0; kb < NKB && ok; ++kb) {
          ok = mbar_wait(bars + 8 * stage, ph, a.status, 12);
          tc_fence_after();
          const uint32_t sa = sbase + stage * FC_STAGE_BYTES, sb = sa + FC_A_BYTES;
#pragma unroll
          for (int ks = 0; ks < FC_BK / 16; ++ks)
            umma(tmem + acc_i * 64, umma_desc_sw128(sa + ks * 32), umma_desc(sb + 2 * ks * 1024, 1024, 128), idesc, (kb | ks) != 0);
          umma_commit(bars + 48 + 8 * stage);
          if (++stage == FC_STAGES) { stage = 0; ph ^= 1; }
        }
        umma_commit(bars + 96 + 8 * acc_i);
        if (++acc_i == 2) { acc_i = 0; aph ^= 1; }
      }
    }
  } else {  // ===== epilogue warps 2..5: TMEM lane quadrant = warp % 4
    const int q = warp & 3, row = q * 32 + lane;
    uint32_t acc_i = 0, aph = 0;
    bool ok = true;
    for (long long it = blockIdx.x; it < total && ok; it += gridDim.x) {
      const int s = (int)(it / a.ntile128), tile = (int)(it % a.ntile128);
      const float* tail = reinterpret_cast<const float*>(a.blob + (long long)((s + a.img_phase) / a.img_per) * a.blob_stride + BLOB_TAIL);
      ok = mbar_wait(bars + 96 + 8 * acc_i, aph, a.status, 13);
      tc_fence_after();
      float acc[4][16];
#pragma unroll
      for (int g = 0; g < 4; ++g) tmem_ld16(tmem + ((uint32_t)(q * 32) << 16) + acc_i * 64 + g * 16, acc[g]);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(bars + 112 + 8 * acc_i);  // accumulator drained: the issuer may reuse it
      const int gw = tile * 128 + row;
      float o0 = __ldg(tail + 192), o1 = __ldg(tail + 193);
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        KeepBits kb = {};
        if (DROP && !a.drop.ptr)  // 16 keep decisions of outputs 16g .. 16g+15: one Philox block
          kb = keep_bits(philox_block_mask(a.drop.seed, a.drop.kind, a.drop.site, a.drop.sample0 + s, a.drop.window0 + gw, g),
                         keep_threshold(a.keep));
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int n = g * 16 + j;
          float h = fmaxf(acc[g][j] + __ldg(tail + n), 0.f);
          if (DROP) {
            if (gw < a.B) {
              const bool keep = a.drop.ptr ? a.drop.ptr[((long long)s * a.B + gw) * 64 + n] != 0.f
                                           : keep_at(kb, j);
              h = keep ? h / a.keep : 0.f;
            }
          }
          o0 = fmaf(h, __ldg(tail + 64 + n), o0);
          o1 = fmaf(h, __ldg(tail + 128 + n), o1);
        }
      }
      if (gw < a.B) {
        o0 = o0 > 20.f ? o0 : log1pf(expf(o0));
        o1 = o1 > 20.f ? o1 : log1pf(expf(o1));
        float2 r = make_float2(o0 > 1e-9f ? o0 : 1e-9f, o1 > 1e-9f ? o1 : 1e-9f);
        *reinterpret_cast<float2*>(a.out + ((long long)s * a.B + gw) * 2) = r;
      }
      if (++acc_i == 2) { acc_i = 0; aph ^= 1; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 128);
}

#include "brl_tc_linear.cuh"
#include "brl_tc_convd3.cuh"

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
TcState* tc_create(int net) {
  TcState* st = new TcState();
  st->net = net;
  st->status = nullptr;
  st->sm_count = 148;
  const NetSpec& n = get_net(net);
  for (int l = 0; l < (net == BRL_NET_LINEAR ? 5 : net == BRL_NET_CONV ? 4 : 12); ++l) { st->loff[l][0] = n.layers[l].w_off; st->loff[l][1] = n.layers[l].b_off; }
  int dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&st->sm_count, cudaDevAttrMultiProcessorCount, dev);
  if (cudaMalloc(&st->status, sizeof(int)) != cudaSuccess) { st->status = nullptr; return st; }
  cudaMemset(st->status, 0, sizeof(int));
  cudaFuncSetAttribute(tc_conv_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, CONV_SMEM);
  cudaFuncSetAttribute(tc_conv_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, CONV_SMEM);
  cudaFuncSetAttribute(tc_fc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FC_SMEM);
  cudaFuncSetAttribute(tc_fc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, FC_SMEM);
  cudaFuncSetAttribute(tcl_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, lin::SMEM);
  cudaFuncSetAttribute(tcc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, cd3::SMEM);
  return st;
}
void tc_destroy(TcState* s) {
  if (!s) return;
  if (s->status) cudaFree(s->status);
  for (auto& v : s->evs)
    for (auto& e : v) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
  delete s;
}
void tc_timing(TcState* s, bool enable) {
  s->timing = enable;
  s->ev_used[0] = s->ev_used[1] = 0;
}
void tc_timing_read(TcState* s, double* ms, long long* launches) {
  for (int k = 0; k < 2; ++k) {
    double t = 0.0;
    for (size_t i = 0; i < s->ev_used[k]; ++i) {
      float e = 0.f;
      cudaEventSynchronize(s->evs[k][i].second);
      cudaEventElapsedTime(&e, s->evs[k][i].first, s->evs[k][i].second);
      t += e;
    }
    ms[k] = t;
    launches[k] = (long long)s->ev_used[k];
    s->ev_used[k] = 0;
  }
}
static void tc_time_begin(TcState* st, int k, cudaStream_t stream) {
  if (!st->timing) return;
  if (st->ev_used[k] == st->evs[k].size()) {
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    st->evs[k].emplace_back(e0, e1);
  }
  cudaEventRecord(st->evs[k][st->ev_used[k]].first, stream);
}
static void tc_time_end(TcState* st, int k, cudaStream_t stream) {
  if (st->timing) cudaEventRecord(st->evs[k][st->ev_used[k]++].second, stream);
}
void tc_trace(TcState* s, long long* buf) { s->trace = buf; }
bool tc_capturable(const TcState* s) { return !s || (!s->timing && !s->trace); }
bool tc_available(const TcState* s) { return s && s->status != nullptr; }  // all three nets (the status word exists: sm_100 context)
bool tc_host_pipeline(const TcState* s) { return tc_available(s) && s->net == BRL_NET_INCEPTION; }
int tc_status(const TcState* s) {
  int v = -1;
  if (s && s->status) cudaMemcpy(&v, s->status, sizeof(int), cudaMemcpyDeviceToHost);
  return v;
}
size_t tc_workspace_bytes(const TcState* s, long long B, long long S) {
  if (s && s->net == BRL_NET_LINEAR)  // fp16 window matrix | weight images
    return (size_t)(((B + 127) / 128) * 128 * lin::KX * 2 + S * (long long)lin::IMG_BYTES + 2048);
  if (s && s->net == BRL_NET_CONV)  // per-tile window images | weight images
    return (size_t)(((B + 3) / 4) * (long long)cd3::XQ_BYTES + S * (long long)cd3::IMG_BYTES + 2048);
  const long long nt128 = (B + 127) / 128, npair = ((B + 3) / 4 + 1) / 2;
  return (size_t)(S * (long long)BLOB_BYTES + S * nt128 * 128 * FEAT_ROW_BYTES + 2 * npair * XIMG_TILE_BYTES + 2048);
}

size_t tc_weight_image_bytes() { return BLOB_BYTES; }

static float inv_keep4(float p_dropout) { return p_dropout > 0.f ? 1.0f / (1.0f - p_dropout * 0.25f) : 1.0f; }

const char* tc_pack_weights(TcState* st, const float* weights, long long w_sample_stride, long long n, unsigned char* images,
                            float p_dropout, cudaStream_t stream) {
  if (!tc_host_pipeline(st)) return "bayesrul_b200: prepacked weight images are implemented for the Inception net only";
  PackArgs pa;
  pa.w = weights; pa.w_stride = w_sample_stride; pa.blob = images; pa.inv4 = inv_keep4(p_dropout);
  for (int l = 0; l < 12; ++l) { pa.off[l][0] = st->loff[l][0]; pa.off[l][1] = st->loff[l][1]; }
  tc_pack_kernel<<<dim3((PACK_THREADS_TOTAL + 255) / 256, (unsigned)n), 256, 0, stream>>>(pa);
  count_launch(1);
  return nullptr;
}

typedef CUresult (*TmaEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
// resolved through the runtime so that the library carries no link-time dependency on libcuda.so
static TmaEncodeFn tma_encode_fn() {
  static TmaEncodeFn encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn) return nullptr;
    encode = reinterpret_cast<TmaEncodeFn>(fn);
  }
  return encode;
}

// Linear net: windows -> fp16 matrix, weights -> fp16 images, one persistent launch (brl_tc_linear.cuh)
static const char* tcl_forward(TcState* st, const float* x, long long B, long long S, const float* weights, long long w_sample_stride,
                               float p_dropout, float* out, void* ws, bool pack_x, cudaStream_t stream, int img_per, int img_phase) {
  if (p_dropout > 0.f) return "bayesrul_b200: the Linear net's tensor-core engine has no dropout path (use engine 'simt')";
  const long long nt128 = (B + 127) / 128, Bpad = nt128 * 128;
  unsigned char* x16 = reinterpret_cast<unsigned char*>(ws);
  unsigned char* img = x16 + ((Bpad * lin::KX * 2 + 255) / 256) * 256;
  if (pack_x) {
    tcl_packx_kernel<<<(unsigned)((Bpad * (lin::KX / 8) + 255) / 256), 256, 0, stream>>>(x, x16, (int)B, (int)Bpad);
    count_launch(1);
  }
  LinPackArgs pa;
  pa.w = weights; pa.w_stride = w_sample_stride; pa.img = img;
  for (int l = 0; l < 5; ++l) { pa.w_off[l] = st->loff[l][0]; pa.b_off[l] = st->loff[l][1]; }
  const long long nimg = w_sample_stride ? (img_phase + S - 1) / img_per + 1 : 1;
  tcl_pack_kernel<<<dim3((lin::IMG_HALVES + lin::TAIL_FLOATS + 255) / 256, (unsigned)nimg), 256, 0, stream>>>(pa);
  CUtensorMap xmap;
  {
    TmaEncodeFn encode = tma_encode_fn();
    if (!encode) return "bayesrul_b200: cuTensorMapEncodeTiled is not available from this driver";
    const cuuint64_t gdim[2] = {(cuuint64_t)lin::KX, (cuuint64_t)Bpad};
    const cuuint64_t gstr[1] = {(cuuint64_t)lin::KX * 2};
    const cuuint32_t box[2] = {64, 128};
    const cuuint32_t estr[2] = {1, 1};
    if (encode(&xmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, x16, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
               CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return "bayesrul_b200: cuTensorMapEncodeTiled failed for the window matrix";
  }
  LinArgs la;
  la.img = img; la.img_stride = w_sample_stride ? lin::IMG_BYTES : 0; la.img_per = img_per; la.img_phase = img_phase; la.out = out;
  la.B = (int)B; la.S = (int)S; la.ntile128 = (int)nt128; la.status = st->status;
  const int grid = (int)std::min<long long>(st->sm_count, S * nt128);
  tcl_kernel<<<grid, 128, lin::SMEM, stream>>>(la, xmap);
  count_launch(2);
  return nullptr;
}

// Conv-D3 net: windows -> per-tile fp16 images, weights -> fp16 images, one persistent launch (brl_tc_convd3.cuh)
static const char* tcc_forward(TcState* st, const float* x, long long B, long long S, const float* weights, long long w_sample_stride,
                               float p_dropout, float* out, void* ws, bool pack_x, cudaStream_t stream, int img_per, int img_phase) {
  if (p_dropout > 0.f) return "bayesrul_b200: the Conv-D3 net's tensor-core engine has no dropout path (use engine 'simt')";
  const long long ntile = (B + 3) / 4;
  unsigned char* ximg = reinterpret_cast<unsigned char*>(ws);
  unsigned char* img = ximg + ((ntile * cd3::XQ_BYTES + 255) / 256) * 256;
  if (pack_x) {
    tcc_packx_kernel<<<(unsigned)((ntile * 6 * ROWS + 255) / 256), 256, 0, stream>>>(x, ximg, (int)B, (int)ntile);
    count_launch(1);
  }
  Cd3PackArgs pa;
  pa.w = weights; pa.w_stride = w_sample_stride; pa.img = img;
  for (int l = 0; l < 4; ++l) { pa.w_off[l] = st->loff[l][0]; pa.b_off[l] = st->loff[l][1]; }
  const long long nimg = w_sample_stride ? (img_phase + S - 1) / img_per + 1 : 1;
  tcc_pack_kernel<<<dim3((cd3::IMG_HALVES + cd3::TAIL_FLOATS + 255) / 256, (unsigned)nimg), 256, 0, stream>>>(pa);
  Cd3Args ca;
  ca.ximg = ximg; ca.img = img; ca.img_stride = w_sample_stride ? cd3::IMG_BYTES : 0; ca.img_per = img_per; ca.img_phase = img_phase;
  ca.out = out;
  ca.B = (int)B; ca.S = (int)S; ca.ntile = (int)ntile; ca.status = st->status;
  const int grid = (int)std::min<long long>(2ll * st->sm_count, S * ntile);
  tcc_kernel<<<grid, 128, cd3::SMEM, stream>>>(ca);
  count_launch(2);
  return nullptr;
}

const char* tc_forward(TcState* st, const float* x, long long B, long long S, const float* weights, long long w_sample_stride,
                       float p_dropout, const brl_noise* noise, float* out, void* ws, size_t ws_bytes, bool pack_x,
                       cudaStream_t stream, const unsigned char* prepacked, int img_per, int img_phase) {
  if (!tc_available(st)) return "bayesrul_b200: tensor-core engine unavailable (no sm_100 context)";
  if (ws_bytes < tc_workspace_bytes(st, B, S)) return "bayesrul_b200: workspace too small for the tensor-core engine";
  if (st->net == BRL_NET_LINEAR) {
    if (prepacked) return "bayesrul_b200: prepacked weight images are implemented for the Inception net only";
    return tcl_forward(st, x, B, S, weights, w_sample_stride, p_dropout, out, ws, pack_x, stream, img_per, img_phase);
  }
  if (st->net == BRL_NET_CONV) {
    if (prepacked) return "bayesrul_b200: prepacked weight images are implemented for the Inception net only";
    return tcc_forward(st, x, B, S, weights, w_sample_stride, p_dropout, out, ws, pack_x, stream, img_per, img_phase);
  }
  const long long nt128 = (B + 127) / 128, nt4 = (B + 3) / 4;
  // workspace: window images (independent of S, so later sample chunks of a batch find them again) | blobs | features
  const int ntx = (int)((nt4 + 1) / 2 * 2);
  unsigned char* ximg = reinterpret_cast<unsigned char*>(ws);
  unsigned char* blob = ximg + (((long long)ntx * XIMG_TILE_BYTES + 255) / 256) * 256;
  const long long nblob = w_sample_stride ? (img_phase + S - 1) / img_per + 1 : 1;
  unsigned char* feat = blob + ((S * (long long)BLOB_BYTES + 255) / 256) * 256;
  if (pack_x) {  // the windows are shared by all MC samples: their fp16 chunk images are built once per batch
    tc_packx_kernel<<<(unsigned)(((long long)ntx * 384 + 255) / 256), 256, 0, stream>>>(x, ximg, (int)B, ntx);
    count_launch(1);
  }
  if (prepacked) {
    blob = const_cast<unsigned char*>(prepacked);
  } else {
    PackArgs pa;
    pa.w = weights; pa.w_stride = w_sample_stride; pa.blob = blob; pa.inv4 = inv_keep4(p_dropout);
    for (int l = 0; l < 12; ++l) { pa.off[l][0] = st->loff[l][0]; pa.off[l][1] = st->loff[l][1]; }
    tc_pack_kernel<<<dim3((PACK_THREADS_TOTAL + 255) / 256, (unsigned)nblob), 256, 0, stream>>>(pa);
    count_launch(1);
  }
  const bool drop = p_dropout > 0.f;
  auto nr = [&](int layer) {
    NoiseRef r;
    r.ptr = noise ? noise->drop_mask[layer] : nullptr;
    r.seed = noise ? noise->seed : 0ull;
    r.kind = KIND_DROPOUT; r.site = layer;
    r.sample0 = noise ? (unsigned)noise->sample0 : 0u;
    r.window0 = noise ? (unsigned)noise->window0 : 0u;
    r.dyn = nullptr;
    return r;
  };
  ConvArgs ca;
  ca.ximg = ximg; ca.blob = blob; ca.blob_stride = w_sample_stride ? BLOB_BYTES : 0; ca.feat = feat;
  ca.img_per = img_per; ca.img_phase = img_phase;
  ca.B = (int)B; ca.S = (int)S; ca.ntile4 = (int)nt4; ca.ntile128 = (int)nt128;
  ca.keep4 = drop ? 1.0f - p_dropout * 0.25f : 1.0f;
  for (int l = 0; l < 12; ++l) ca.drop[l] = nr(l);
  {  // key of the native dropout masks (brl_tc_conv.cuh: philox7_rk)
    const unsigned long long seed = noise ? noise->seed : 0ull;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    for (int r = 0; r < 7; ++r) { ca.rk[2 * r] = k0; ca.rk[2 * r + 1] = k1; k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
    ca.sample0 = noise ? (uint32_t)noise->sample0 : 0u;
    ca.window0 = noise ? (uint32_t)noise->window0 : 0u;
    ca.inj_mask = 0u;
    ca.keepT2 = keep_threshold(ca.keep4) * 0x10001u;
    for (int l = 0; l < 12; ++l)
      if (ca.drop[l].ptr) ca.inj_mask |= 1u << l;
  }
  ca.status = st->status;
  ca.trace = st->trace;
  const long long items = S * ((nt4 + 1) / 2);
  static const int env_conv = getenv("BRL_CONV_GRID") ? atoi(getenv("BRL_CONV_GRID")) : 0;  // experiment knobs
  static const int env_fc = getenv("BRL_FC_GRID") ? atoi(getenv("BRL_FC_GRID")) : 0;
  const int grid = (int)std::min<long long>(env_conv > 0 ? env_conv : st->sm_count, items);
  tc_time_begin(st, 0, stream);
  if (drop) tc_conv_kernel<true><<<grid, CONV_THREADS, CONV_SMEM, stream>>>(ca);
  else tc_conv_kernel<false><<<grid, CONV_THREADS, CONV_SMEM, stream>>>(ca);
  tc_time_end(st, 0, stream);
  FcArgs fa;
  fa.blob = blob; fa.blob_stride = ca.blob_stride; fa.img_per = img_per; fa.img_phase = img_phase; fa.out = out;
  fa.B = (int)B; fa.S = (int)S; fa.ntile128 = (int)nt128;
  fa.keep = drop ? 1.0f - p_dropout : 1.0f;
  fa.drop = nr(10);
  fa.status = st->status;
  const int gridf = (int)std::min<long long>(env_fc > 0 ? env_fc : st->sm_count, S * nt128);
  // TMA view of the feature tensor: [S * Bpad rows][2400 fp16], boxes of 128 rows x 64 columns, 128-byte swizzle
  CUtensorMap fmap;
  {
    const cuuint64_t gdim[2] = {2400, (cuuint64_t)(S * nt128 * 128)};
    const cuuint64_t gstr[1] = {FEAT_ROW_BYTES};
    const cuuint32_t box[2] = {FC_BK, 128};
    const cuuint32_t estr[2] = {1, 1};
    TmaEncodeFn encode = tma_encode_fn();  // (no link-time dependency on libcuda.so: the library must load without a driver)
    if (!encode) return "bayesrul_b200: cuTensorMapEncodeTiled is not available from this driver";
    const CUresult r = encode(&fmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, feat, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return "bayesrul_b200: cuTensorMapEncodeTiled failed for the feature tensor";
  }
  tc_time_begin(st, 1, stream);
  if (drop) tc_fc_kernel<true><<<gridf, 192, FC_SMEM, stream>>>(fa, fmap);
  else tc_fc_kernel<false><<<gridf, 192, FC_SMEM, stream>>>(fa, fmap);
  tc_time_end(st, 1, stream);
  count_launch(2);
  return nullptr;
}

}  // namespace brl
