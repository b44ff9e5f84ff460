// fp32 SIMT engine: implicit-GEMM conv / linear layers with the variational rules fused in the
// gather prologue and the epilogue, plus the small reductions of the ELBO / predictive path.
// This is the parity engine (rtol 1e-3 vs the oracle); the tcgen05 engine lives in brl_tc.cu.
#include <atomic>
#include <cstddef>

#include "brl_kernels.cuh"
#include "brl_philox.cuh"

namespace brl {

std::atomic<long long> g_launch_count{0};
long long launch_count() { return g_launch_count.load(); }
void count_launch(int n) { g_launch_count.fetch_add(n); }

// ------------------------------------------------------------------------------------------------
// helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float noise_normal(const NoiseRef& nz, int s, int b, int B, int per_window, int e) {
  if (nz.ptr) return nz.ptr[((long long)s * B + b) * per_window + e];
  const NoiseKey k = noise_key(nz);
  return philox_normal(k.seed, nz.kind, nz.site, k.sample0 + s, k.window0 + b, e);
}
__device__ __forceinline__ float softplusf(float x) { return x > 20.0f ? x : log1pf(expf(x)); }

__device__ __forceinline__ double block_sum(double v) {
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
  return v;  // valid in thread 0
}

// ------------------------------------------------------------------------------------------------
// pooling
// ------------------------------------------------------------------------------------------------
__global__ void maxpool3_kernel(const PoolParams p) {
  const long long total = p.n_img * p.C * p.Hin * p.Win;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int w = i % p.Win;
    const int h = (i / p.Win) % p.Hin;
    const int c = (i / ((long long)p.Win * p.Hin)) % p.C;
    const long long img = i / ((long long)p.Win * p.Hin * p.C);
    const float* src = p.in + img * p.in_img_stride + (long long)c * p.sC + (long long)w * p.sW;
    float v = src[(long long)h * p.sH];
    if (h > 0) v = fmaxf(v, src[(long long)(h - 1) * p.sH]);
    if (h + 1 < p.Hin) v = fmaxf(v, src[(long long)(h + 1) * p.sH]);
    p.out[img * p.out_img_stride + ((long long)c * p.Hin + h) * p.Win + w] = v;
  }
}
void launch_maxpool3(const PoolParams& p, cudaStream_t st) {
  const long long total = p.n_img * p.C * p.Hin * p.Win;
  ++g_launch_count;
  maxpool3_kernel<<<(unsigned)min((total + 255) / 256, (long long)148 * 16), 256, 0, st>>>(p);
}

__device__ __forceinline__ int argmax3_first(const float* src, int o, int H, long long sH) {
  int best = o > 0 ? o - 1 : o;
  float bv = src[(long long)best * sH];
  for (int t = best + 1; t <= min(o + 1, H - 1); ++t) {
    const float v = src[(long long)t * sH];
    if (v > bv) { bv = v; best = t; }
  }
  return best;
}
__global__ void maxpool3_bwd_kernel(const PoolParams p, const float* gout, float* gin) {
  const long long total = p.n_img * p.C * p.Hin * p.Win;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int w = i % p.Win;
    const int h = (i / p.Win) % p.Hin;
    const int c = (i / ((long long)p.Win * p.Hin)) % p.C;
    const long long img = i / ((long long)p.Win * p.Hin * p.C);
    const float* src = p.in + img * p.in_img_stride + (long long)c * p.sC + (long long)w * p.sW;
    const float* go = gout + img * p.out_img_stride + (long long)c * p.Hin * p.Win + w;
    float g = 0.f;
    for (int o = max(h - 1, 0); o <= min(h + 1, p.Hin - 1); ++o)
      if (argmax3_first(src, o, p.Hin, p.sH) == h) g += go[(long long)o * p.Win];
    atomicAdd(gin + img * p.in_img_stride + (long long)c * p.sC + (long long)h * p.sH + (long long)w * p.sW, g);
  }
}
void launch_maxpool3_bwd(const PoolParams& p, const float* gout, float* gin, cudaStream_t st) {
  const long long total = p.n_img * p.C * p.Hin * p.Win;
  ++g_launch_count;
  maxpool3_bwd_kernel<<<(unsigned)min((total + 255) / 256, (long long)148 * 16), 256, 0, st>>>(p, gout, gin);
}

__global__ void avgpool2_kernel(const PoolParams p) {
  const long long total = p.n_img * p.C * p.Hout * p.Win;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int w = i % p.Win;
    const int h = (i / p.Win) % p.Hout;
    const int c = (i / ((long long)p.Win * p.Hout)) % p.C;
    const long long img = i / ((long long)p.Win * p.Hout * p.C);
    const float* src = p.in + img * p.in_img_stride + (long long)c * p.sC + (long long)w * p.sW;
    p.out[img * p.out_img_stride + ((long long)c * p.Hout + h) * p.Win + w] =
        0.5f * (src[(long long)(2 * h) * p.sH] + src[(long long)(2 * h + 1) * p.sH]);
  }
}
void launch_avgpool2(const PoolParams& p, cudaStream_t st) {
  const long long total = p.n_img * p.C * p.Hout * p.Win;
  ++g_launch_count;
  avgpool2_kernel<<<(unsigned)min((total + 255) / 256, (long long)148 * 16), 256, 0, st>>>(p);
}
__global__ void avgpool2_bwd_kernel(const PoolParams p, const float* gout, float* gin) {
  const long long total = p.n_img * p.C * p.Hin * p.Win;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int w = i % p.Win;
    const int h = (i / p.Win) % p.Hin;
    const int c = (i / ((long long)p.Win * p.Hin)) % p.C;
    const long long img = i / ((long long)p.Win * p.Hin * p.C);
    if (h < 2 * p.Hout)
      gin[img * p.in_img_stride + (long long)c * p.sC + (long long)h * p.sH + (long long)w * p.sW] +=
          0.5f * gout[img * p.out_img_stride + ((long long)c * p.Hout + (h >> 1)) * p.Win + w];
  }
}
void launch_avgpool2_bwd(const PoolParams& p, const float* gout, float* gin, cudaStream_t st) {
  const long long total = p.n_img * p.C * p.Hin * p.Win;
  ++g_launch_count;
  avgpool2_bwd_kernel<<<(unsigned)min((total + 255) / 256, (long long)148 * 16), 256, 0, st>>>(p, gout, gin);
}

// ------------------------------------------------------------------------------------------------
// backward through activation / dropout / head
// ------------------------------------------------------------------------------------------------
__global__ void bwd_act_kernel(const BwdAct p) {
  const long long per = (long long)p.N * p.P, total = p.n_img * per;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long img = i / per;
    const int e = (int)(i - img * per);
    const int n = e / p.P, pp = e - n * p.P;
    const long long oidx = img * p.img_stride + (long long)(p.co_off + n) * p.out_P + pp;
    const float g = p.gout[oidx], o = p.outv[oidx];
    float d;
    if (p.head) d = o > 1e-9f ? g * (1.0f - expf(-o)) : 0.f;
    else if (p.relu) d = o > 0.f ? g * p.inv_keep : 0.f;
    else d = g * p.inv_keep;
    p.dpre[i] = d;
    const int s = (int)(img / p.B), b = (int)(img - (long long)s * p.B);
    if (p.dvar) {
      const float sd = p.sd[i];
      const float eps = noise_normal(p.eps, s, b, p.B, (int)per, e);
      p.dvar[i] = sd > 0.f ? d * eps / (2.0f * sd) : 0.f;
    }
    if (p.dpert) p.dpert[i] = d * p.sign_out[img * p.N + n];
  }
}
void launch_bwd_act(const BwdAct& p, cudaStream_t st) {
  const long long total = p.n_img * p.N * p.P;
  ++g_launch_count;
  bwd_act_kernel<<<(unsigned)min((total + 255) / 256, (long long)148 * 16), 256, 0, st>>>(p);
}

// ------------------------------------------------------------------------------------------------
// guide samplers
// ------------------------------------------------------------------------------------------------
__global__ void sample_normal_kernel(const float* __restrict__ mu, const float* __restrict__ sigma, long long P,
                                     NoiseRef eps, float* __restrict__ w, float* __restrict__ delta, long long mu_stride,
                                     int sample_stride, int per, int phase) {
  const long long nblk = (P + 3) >> 2;
  const int s = blockIdx.y, se = s * sample_stride;  // draw s: MC-sample index / injected row sample0 + se
  mu += (long long)((s + phase) / per) * mu_stride;
  sigma += (long long)((s + phase) / per) * mu_stride;
  for (long long blk = blockIdx.x * (long long)blockDim.x + threadIdx.x; blk < nblk; blk += (long long)gridDim.x * blockDim.x) {
    float z[4];
    const long long e0 = blk << 2;
    if (eps.ptr) {
#pragma unroll
      for (int l = 0; l < 4; ++l) z[l] = e0 + l < P ? eps.ptr[(long long)se * P + e0 + l] : 0.f;
    } else {
      const NoiseKey k = noise_key(eps);
      const float4 n4 = normal4(philox_block(k.seed, KIND_WEIGHT_EPS, 0, k.sample0 + se, 0, (uint32_t)blk));
      z[0] = n4.x; z[1] = n4.y; z[2] = n4.z; z[3] = n4.w;
    }
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      const long long e = e0 + l;
      if (e < P) {
        w[(long long)s * P + e] = fmaf(sigma[e], z[l], mu[e]);
        if (delta) delta[(long long)s * P + e] = z[l];
      }
    }
  }
}
void launch_sample_normal(const float* mu, const float* sigma, long long P, long long S, NoiseRef eps, float* w,
                          float* delta, cudaStream_t st, long long mu_stride, int sample_stride, int per, int phase) {
  const long long nblk = (P + 3) >> 2;
  dim3 grid((unsigned)min((nblk + 255) / 256, (long long)148 * 8), (unsigned)S);
  ++g_launch_count;
  sample_normal_kernel<<<grid, 256, 0, st>>>(mu, sigma, P, eps, w, delta, mu_stride, sample_stride, per, phase);
}

// The radial guide needs ||eps|| over each whole site before any weight of the site exists, so the draw is two passes over
// the same Philox stream (the stream of sample_normal_kernel: block = element >> 2, four normals per block).
__device__ __forceinline__ void weight_eps4(const NoiseRef& eps, const NoiseKey& k, int s, long long P, long long blk, float (&z)[4]) {
  const long long e0 = blk << 2;
  if (eps.ptr) {
#pragma unroll
    for (int l = 0; l < 4; ++l) z[l] = e0 + l < P ? eps.ptr[(long long)s * P + e0 + l] : 0.f;
  } else {
    const float4 n4 = normal4(philox_block(k.seed, KIND_WEIGHT_EPS, 0, k.sample0 + s, 0, (uint32_t)blk));
    z[0] = n4.x; z[1] = n4.y; z[2] = n4.z; z[3] = n4.w;
  }
}
__global__ void radial_norm_kernel(long long P, const long long* __restrict__ site_off, int n_sites, NoiseRef eps,
                                   float* __restrict__ norms, int sample_stride) {
  const int j = blockIdx.x, s = blockIdx.y, se = s * sample_stride;
  const long long beg = site_off[j], end = site_off[j + 1];
  const NoiseKey k = noise_key(eps);
  double acc = 0.0;
  for (long long blk = (beg >> 2) + threadIdx.x; blk <= ((end - 1) >> 2); blk += blockDim.x) {
    float z[4];
    weight_eps4(eps, k, se, P, blk, z);
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      const long long e = (blk << 2) + l;
      if (e >= beg && e < end) acc += (double)z[l] * z[l];
    }
  }
  acc = block_sum(acc);
  if (threadIdx.x == 0) norms[(long long)s * n_sites + j] = (float)sqrt(acc);
}
__global__ void radial_apply_kernel(const float* __restrict__ mu, const float* __restrict__ sigma, long long P,
                                    const long long* __restrict__ site_off, int n_sites, NoiseRef eps, NoiseRef r,
                                    const float* __restrict__ norms, float* __restrict__ w, float* __restrict__ delta,
                                    long long mu_stride, int sample_stride, int per, int phase) {
  const int s = blockIdx.y, se = s * sample_stride;
  mu += (long long)((s + phase) / per) * mu_stride;
  sigma += (long long)((s + phase) / per) * mu_stride;
  const long long nblk = (P + 3) >> 2;
  const NoiseKey k = noise_key(eps), rk = noise_key(r);
  for (long long blk = blockIdx.x * (long long)blockDim.x + threadIdx.x; blk < nblk; blk += (long long)gridDim.x * blockDim.x) {
    float z[4];
    weight_eps4(eps, k, se, P, blk, z);
    const long long e0 = blk << 2;
    int lo = 0, hi = n_sites - 1;  // site of e0: last j with site_off[j] <= e0
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (site_off[mid] <= e0) lo = mid; else hi = mid - 1;
    }
    int j = lo;
    float scale = 0.f;
    bool have = false;
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      const long long e = e0 + l;
      if (e >= P) break;
      while (e >= site_off[j + 1]) { ++j; have = false; }
      if (!have) {
        const float rr = r.ptr ? r.ptr[(long long)se * n_sites + j]
                               : philox_normal(rk.seed, KIND_RADIAL_R, 0, rk.sample0 + se, 0, (uint32_t)j);
        scale = rr / norms[(long long)s * n_sites + j];
        have = true;
      }
      const float d = z[l] * scale;
      w[(long long)s * P + e] = fmaf(d, sigma[e], mu[e]);
      if (delta) delta[(long long)s * P + e] = d;
    }
  }
}
void launch_sample_radial(const float* mu, const float* sigma, long long P, long long S, const long long* site_off,
                          int n_sites, int max_site, NoiseRef eps, NoiseRef r, float* norms, float* w, float* delta,
                          cudaStream_t st, long long mu_stride, int sample_stride, int per, int phase) {
  ++g_launch_count;
  radial_norm_kernel<<<dim3(n_sites, (unsigned)S), 256, 0, st>>>(P, site_off, n_sites, eps, norms, sample_stride);
  ++g_launch_count;
  const long long nblk = (P + 3) >> 2;
  radial_apply_kernel<<<dim3((unsigned)min((nblk + 255) / 256, (long long)148 * 8), (unsigned)S), 256, 0, st>>>(
      mu, sigma, P, site_off, n_sites, eps, r, norms, w, delta, mu_stride, sample_stride, per, phase);
}

__global__ void gen_signs_kernel(float* dst, long long S, long long B, int C, NoiseRef nz) {
  const long long total = S * B * C;
  const NoiseKey k = noise_key(nz);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = i % C;
    const long long sb = i / C;
    const int b = sb % B, s = sb / B;
    dst[i] = philox_sign(k.seed, nz.kind, nz.site, k.sample0 + s, k.window0 + b, c);
  }
}
__global__ void gen_signs_multi_kernel(const SignJobs jobs, long long B, NoiseRef base, int sample_stride) {
  const long long total = jobs.start[jobs.n];
  const int m = blockIdx.y;  // member: its tensors [B, C] follow the previous member's, MC-sample index + m sample_stride
  NoiseKey k = noise_key(base);
  k.sample0 += (unsigned)(m * sample_stride);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int j = 0;
    while (j + 1 < jobs.n && i >= jobs.start[j + 1]) ++j;
    // one work item = one Philox block = the signs of four consecutive channels of a window (element c: block c >> 2, lane c & 3,
    // the keying of philox_sign)
    const long long e = i - jobs.start[j];
    const int C = jobs.C[j], Q = (C + 3) >> 2, q = (int)(e % Q), b = (int)(e / Q);
    const uint4 r = philox_block(k.seed, jobs.kind[j], jobs.site[j], k.sample0, k.window0 + b, (uint32_t)q);
    float* d = jobs.dst[j] + ((long long)m * B + b) * C + 4 * q;
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int l = 0; l < 4; ++l)
      if (4 * q + l < C) d[l] = (w[l] >> 31) ? -1.0f : 1.0f;
  }
}
void launch_gen_signs_multi(const SignJobs& jobs, long long B, NoiseRef base, cudaStream_t st, int members, int sample_stride) {
  const long long total = jobs.start[jobs.n];
  if (total <= 0) return;
  ++g_launch_count;
  gen_signs_multi_kernel<<<dim3((unsigned)min((total + 255) / 256, (long long)148 * 8), (unsigned)members), 256, 0, st>>>(
      jobs, B, base, sample_stride);
}
void launch_gen_signs(float* dst, long long S, long long B, int C, NoiseRef nz, cudaStream_t st) {
  const long long total = S * B * C;
  ++g_launch_count;
  gen_signs_kernel<<<(unsigned)min((total + 255) / 256, (long long)148 * 8), 256, 0, st>>>(dst, S, B, C, nz);
}

// ------------------------------------------------------------------------------------------------
// likelihoods
// ------------------------------------------------------------------------------------------------
__global__ void nll_elbo_kernel(const float* __restrict__ out, const float* __restrict__ y, long long B, float gscale,
                                double* acc, float* __restrict__ gout) {
  double nll = 0.0, se = 0.0;
  for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
    const float loc = out[2 * b], sc = out[2 * b + 1];
    const float s = softplusf(sc);  // second softplus: positive_scale=False (bayesian.py:73-76)
    const float d = y[b] - loc, r = d / s;
    nll += 0.5 * (double)r * r + (double)logf(s) + 0.9189385332046727;
    se += (double)d * d;
    if (gout) {
      const float sig = sc > 20.0f ? 1.0f : 1.0f / (1.0f + expf(-sc));
      gout[2 * b] = -r / s * gscale;
      gout[2 * b + 1] = (1.0f - r * r) / s * sig * gscale;
    }
  }
  nll = block_sum(nll);
  se = block_sum(se);
  if (threadIdx.x == 0) {
    atomicAdd(acc + 0, nll);
    atomicAdd(acc + 1, se);
  }
}
void launch_nll_elbo(const float* out, const float* y, long long B, float gscale, double* acc, float* gout,
                     cudaStream_t st) {
  ++g_launch_count;
  nll_elbo_kernel<<<(unsigned)min((B + 255) / 256, (long long)148), 256, 0, st>>>(out, y, B, gscale, acc, gout);
}

__global__ void nll_hnn_kernel(const float* __restrict__ out, const float* __restrict__ y, long long B, double* acc,
                               float* __restrict__ gout) {
  double loss = 0.0, se = 0.0;
  const float invB = 1.0f / (float)B;
  for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
    const float loc = out[2 * b], sc = out[2 * b + 1];
    const float var0 = sc * sc, var = fmaxf(var0, 1e-6f);  // F.gaussian_nll_loss eps clamp
    const float d = loc - y[b];
    loss += 0.5 * ((double)logf(var) + (double)d * d / var);
    se += (double)d * d;
    if (gout) {
      gout[2 * b] = d / var * invB;
      gout[2 * b + 1] = var0 > 1e-6f ? 0.5f * (1.0f / var - d * d / (var * var)) * 2.0f * sc * invB : 0.f;
    }
  }
  loss = block_sum(loss);
  se = block_sum(se);
  if (threadIdx.x == 0) {
    atomicAdd(acc + 0, loss / (double)B);
    atomicAdd(acc + 1, se / (double)B);
  }
}
void launch_nll_hnn(const float* out, const float* y, long long B, double* acc, float* gout, cudaStream_t st) {
  ++g_launch_count;
  nll_hnn_kernel<<<(unsigned)min((B + 255) / 256, (long long)148), 256, 0, st>>>(out, y, B, acc, gout);
}

// ------------------------------------------------------------------------------------------------
// KL + gradient finalisation
// ------------------------------------------------------------------------------------------------
// member blockIdx.y: its parameters, draws and gradients P floats after the previous member's, its KL at kl_acc + m kl_stride
__device__ __forceinline__ Finalize member_finalize(Finalize p) {
  const long long o = p.P * blockIdx.y;
  auto sh = [o](auto* q) { return q ? q + o : q; };
  p.mu = sh(p.mu); p.sigma = sh(p.sigma); p.w = sh(p.w); p.delta = sh(p.delta); p.g0 = sh(p.g0); p.g1 = sh(p.g1);
  p.grad_mu = sh(p.grad_mu); p.grad_sigma = sh(p.grad_sigma); p.grad_log_sigma = sh(p.grad_log_sigma);
  p.kl_acc += (long long)p.kl_stride * blockIdx.y;
  return p;
}
__global__ void finalize_kernel(const Finalize p_) {
  const Finalize p = member_finalize(p_);
  double kl = 0.0;
  const float isp2 = 1.0f / (p.prior_scale * p.prior_scale);
  const float lsp = logf(p.prior_scale);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < p.P; i += (long long)gridDim.x * blockDim.x) {
    const float mu = p.mu[i], sg = p.sigma[i];
    float gmu = 0.f, gsg = 0.f, dmu_kl, dsg_kl;
    if (p.guide == 1) {  // radial: sampled log q - log p (Trace_ELBO)
      const float w = p.w[i], d = p.delta[i];
      const float zp = (w - p.prior_loc) / p.prior_scale;
      kl += (double)(-logf(sg) - 0.5f * d * d) - (double)(-lsp - 0.5f * zp * zp);
      dmu_kl = (w - p.prior_loc) * isp2;
      dsg_kl = -1.0f / sg + (w - p.prior_loc) * isp2 * d;
      if (p.g0) { gmu = p.g0[i]; gsg = p.g0[i] * d; }
    } else {
      const float dm = mu - p.prior_loc;
      kl += (double)(lsp - logf(sg)) + (double)((sg * sg + dm * dm) * 0.5f * isp2) - 0.5;
      dmu_kl = dm * isp2;
      dsg_kl = -1.0f / sg + sg * isp2;
      if (p.g0) {
        gmu = p.g0[i];
        if (p.mode == 2) gsg = 2.0f * sg * p.g1[i];       // LRT: d/dsigma through sigma^2
        else if (p.mode == 3) gsg = p.g1[i] * p.delta[i]; // flipout: dDeltaW * eps
        else gsg = p.g0[i] * p.delta[i];                   // weight sampling
      }
    }
    if (p.grad_mu) {
      gmu = fmaf(p.c_kl, dmu_kl, gmu);
      gsg = fmaf(p.c_kl, dsg_kl, gsg);
      if (!p.first) { gmu += p.grad_mu[i]; gsg += p.grad_sigma[i]; }
      p.grad_mu[i] = gmu;
      p.grad_sigma[i] = gsg;
      if (p.grad_log_sigma) p.grad_log_sigma[i] = gsg * sg;
    }
  }
  kl = block_sum(kl);
  if (threadIdx.x == 0) atomicAdd(p.kl_acc, kl);
}
void launch_finalize(const Finalize& p, cudaStream_t st) {
  ++g_launch_count;
  finalize_kernel<<<dim3((unsigned)min((p.P + 255) / 256, (long long)148 * 4), (unsigned)max(1, p.members)), 256, 0, st>>>(p);
}

__global__ void post_scalars_kernel(double* scalars, const double* acc, double c_nll, double c, int particles,
                                    long long B) {
  // acc = {nll_sum over particles, squared error sum over particles, kl sum over particles}; member m (thread m): [m][4]
  scalars += 4 * threadIdx.x;
  acc += 4 * threadIdx.x;
  scalars[0] = (c_nll * acc[0] + c * acc[2]) / particles;
  scalars[1] = acc[0] / particles;
  scalars[2] = acc[2] / particles;
  scalars[3] = acc[1] / ((double)particles * (double)B);
}
void launch_post_scalars(double* scalars, const double* acc, double c_nll, double c, int particles, long long B,
                         cudaStream_t st, int members) {
  ++g_launch_count;
  post_scalars_kernel<<<1, members, 0, st>>>(scalars, acc, c_nll, c, particles, B);
}

__global__ void log_sigma_grad_kernel(const float* gs, const float* sigma, float* gls, long long P) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < P; i += (long long)gridDim.x * blockDim.x)
    gls[i] = gs[i] * sigma[i];
}
void launch_log_sigma_grad(const float* gs, const float* sigma, float* gls, long long P, cudaStream_t st) {
  ++g_launch_count;
  log_sigma_grad_kernel<<<(unsigned)min((P + 255) / 256, (long long)148 * 4), 256, 0, st>>>(gs, sigma, gls, P);
}

// ------------------------------------------------------------------------------------------------
// predictive moments (Welford over MC samples; chunks merge through `state`)
// ------------------------------------------------------------------------------------------------
__global__ void moments_update_kernel(const float* __restrict__ out, long long S, long long B, float* state, int first) {
  for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
    float n = 0.f, mean = 0.f, m2 = 0.f, s2 = 0.f;
    if (!first) { n = state[b]; mean = state[B + b]; m2 = state[2 * B + b]; s2 = state[3 * B + b]; }
    // the loads do not depend on the Welford chain: batches of 16 are issued ahead of it (the loop was one DRAM round trip per MC
    // sample: 52 us for S = 100); the arithmetic and its order are unchanged
    long long s = 0;
    for (; s + 16 <= S; s += 16) {
      float2 o[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) o[u] = __ldcs(reinterpret_cast<const float2*>(out + ((s + u) * B + b) * 2));
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        n += 1.f;
        const float d = o[u].x - mean;
        mean += d / n;
        m2 = fmaf(d, o[u].x - mean, m2);
        s2 = fmaf(o[u].y, o[u].y, s2);
      }
    }
    for (; s < S; ++s) {
      const float2 o = *reinterpret_cast<const float2*>(out + (s * B + b) * 2);
      n += 1.f;
      const float d = o.x - mean;
      mean += d / n;
      m2 = fmaf(d, o.x - mean, m2);
      s2 = fmaf(o.y, o.y, s2);
    }
    state[b] = n; state[B + b] = mean; state[2 * B + b] = m2; state[3 * B + b] = s2;
  }
}
void launch_moments_update(const float* out, long long S, long long B, float* state, int first, cudaStream_t st) {
  ++g_launch_count;
  moments_update_kernel<<<(unsigned)min((B + 127) / 128, (long long)148 * 8), 128, 0, st>>>(out, S, B, state, first);
}
__global__ void moments_final_kernel(const float* __restrict__ state, long long B, float* pred, float* std, float* ep,
                                     float* al) {
  for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
    const float n = state[b];
    const float e = state[2 * B + b] / (n - 1.f);  // unbiased: loc.var(0) (bayesian.py:212)
    const float a = state[3 * B + b] / n;
    pred[b] = state[B + b];
    if (ep) ep[b] = e;
    if (al) al[b] = a;
    std[b] = sqrtf(a + e);
  }
}
void launch_moments_final(const float* state, long long B, float* pred, float* std, float* ep, float* al,
                          cudaStream_t st) {
  ++g_launch_count;
  moments_final_kernel<<<(unsigned)min((B + 255) / 256, (long long)148 * 8), 256, 0, st>>>(state, B, pred, std, ep, al);
}

// Samples [j0, j0 + sc) of the member-major sample axis j = m S + s of brl_predict_moments_ensemble (out [sc,B,2]): member
// m = j0 / S + blockIdx.y takes its segment of the chunk, a sequential Welford into its own state [4,B] in the arithmetic
// order of moments_update_kernel (a member whose first sample is in the chunk starts from zero)
__global__ void moments_update_members_kernel(const float* __restrict__ out, long long j0, long long sc, long long S, long long B,
                                              float* state /*[M,4,B]*/) {
  const long long m = j0 / S + blockIdx.y;
  const long long lo = max(j0, m * S), hi = min(j0 + sc, (m + 1) * S), ns = hi - lo;
  const bool first = lo == m * S;
  out += (lo - j0) * B * 2;
  state += m * 4 * B;
  for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
    float n = 0.f, mean = 0.f, m2 = 0.f, s2 = 0.f;
    if (!first) { n = state[b]; mean = state[B + b]; m2 = state[2 * B + b]; s2 = state[3 * B + b]; }
    long long s = 0;
    for (; s + 16 <= ns; s += 16) {
      float2 o[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) o[u] = __ldcs(reinterpret_cast<const float2*>(out + ((s + u) * B + b) * 2));
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        n += 1.f;
        const float d = o[u].x - mean;
        mean += d / n;
        m2 = fmaf(d, o[u].x - mean, m2);
        s2 = fmaf(o[u].y, o[u].y, s2);
      }
    }
    for (; s < ns; ++s) {
      const float2 o = *reinterpret_cast<const float2*>(out + (s * B + b) * 2);
      n += 1.f;
      const float d = o.x - mean;
      mean += d / n;
      m2 = fmaf(d, o.x - mean, m2);
      s2 = fmaf(o.y, o.y, s2);
    }
    state[b] = n; state[B + b] = mean; state[2 * B + b] = m2; state[3 * B + b] = s2;
  }
}
void launch_moments_update_members(const float* out, long long j0, long long sc, long long S, long long B, float* state,
                                   cudaStream_t st) {
  const long long members = (j0 + sc - 1) / S - j0 / S + 1;
  ++g_launch_count;
  moments_update_members_kernel<<<dim3((unsigned)min((B + 127) / 128, (long long)148 * 8), (unsigned)members), 128, 0, st>>>(
      out, j0, sc, S, B, state);
}
// state [M,4,B] -> out [4,M,B] = (pred, std, ep_var, al_var), the arithmetic of moments_final_kernel
__global__ void moments_final_members_kernel(const float* __restrict__ state, long long M, long long B, float* out) {
  const long long MB = M * B;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < MB; i += (long long)gridDim.x * blockDim.x) {
    const long long m = i / B, b = i % B;
    const float* st = state + m * 4 * B;
    const float n = st[b];
    const float e = st[2 * B + b] / (n - 1.f);
    const float a = st[3 * B + b] / n;
    out[i] = st[B + b];
    out[2 * MB + i] = e;
    out[3 * MB + i] = a;
    out[MB + i] = sqrtf(a + e);
  }
}
void launch_moments_final_members(const float* state, long long M, long long B, float* out, cudaStream_t st) {
  ++g_launch_count;
  moments_final_members_kernel<<<(unsigned)min((M * B + 255) / 256, (long long)148 * 8), 256, 0, st>>>(state, M, B, out);
}

__global__ void moments_direct_kernel(const float* __restrict__ out, long long S, long long B, float* pred, float* std,
                                      float* ep, float* al) {
  for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
    float n = 0.f, mean = 0.f, m2 = 0.f, s2 = 0.f;
    for (long long s = 0; s < S; ++s) {
      const float2 o = *reinterpret_cast<const float2*>(out + (s * B + b) * 2);
      n += 1.f;
      const float d = o.x - mean;
      mean += d / n;
      m2 = fmaf(d, o.x - mean, m2);
      s2 = fmaf(o.y, o.y, s2);
    }
    const float e = m2 / (n - 1.f), a = s2 / n;
    pred[b] = mean; ep[b] = e; al[b] = a; std[b] = sqrtf(a + e);
  }
}
void launch_moments_direct(const float* out, long long S, long long B, float* pred, float* std, float* ep, float* al,
                           cudaStream_t st) {
  ++g_launch_count;
  moments_direct_kernel<<<(unsigned)min((B + 127) / 128, (long long)148 * 8), 128, 0, st>>>(out, S, B, pred, std, ep, al);
}

__global__ void aggregate_kernel(const float* __restrict__ out, long long S, long long B, float* agg) {
  for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
    float n = 0.f, mean = 0.f, m2 = 0.f, s2 = 0.f, wl = 0.f, wp = 0.f;
    for (long long s = 0; s < S; ++s) {
      const float2 o = *reinterpret_cast<const float2*>(out + (s * B + b) * 2);
      n += 1.f;
      const float d = o.x - mean;
      mean += d / n;
      m2 = fmaf(d, o.x - mean, m2);
      s2 = fmaf(o.y, o.y, s2);
      const float prec = 1.0f / (o.y * o.y);
      wl = fmaf(o.x, prec, wl);
      wp += prec;
    }
    const float sc = sqrtf(s2 / n + m2 / (n - 1.f));
    agg[2 * b] = wl / wp;
    agg[2 * b + 1] = sc + logf(-expm1f(-sc));  // inverse softplus (positive_scale=False)
  }
}
void launch_aggregate(const float* out, long long S, long long B, float* agg, cudaStream_t st) {
  ++g_launch_count;
  aggregate_kernel<<<(unsigned)min((B + 127) / 128, (long long)148 * 8), 128, 0, st>>>(out, S, B, agg);
}

__global__ void mixture_kernel(const float* __restrict__ mu_m, const float* __restrict__ sd_m, long long M, long long n,
                               float* mu, float* sd) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    double a = 0.0, q = 0.0;
    for (long long m = 0; m < M; ++m) {
      const double u = mu_m[m * n + i], s = sd_m[m * n + i];
      a += u;
      q += u * u + s * s;
    }
    a /= (double)M;
    mu[i] = (float)a;
    sd[i] = (float)sqrt(q / (double)M - a * a);  // biased mixture variance (deepens.py:24)
  }
}
void launch_mixture(const float* mu_m, const float* sd_m, long long M, long long n, float* mu, float* sd,
                    cudaStream_t st) {
  ++g_launch_count;
  mixture_kernel<<<(unsigned)min((n + 255) / 256, (long long)148 * 8), 256, 0, st>>>(mu_m, sd_m, M, n, mu, sd);
}

// ------------------------------------------------------------------------------------------------
// test-time scalar metrics (bayesian.py:217-224; results/metrics.py:210-274)
// ------------------------------------------------------------------------------------------------
// member m = blockIdx.y (grid.y = M) of [M,n] inputs: its scratch is the m-th 1024 bytes (hist[100] u32, acc[3] doubles at +512 B)
__global__ void test_metrics_acc_kernel(const float* __restrict__ pred, const float* __restrict__ std,
                                        const float* __restrict__ y, long long n, unsigned int* hist) {
  const long long m = blockIdx.y;
  pred += m * n;
  std += m * n;
  y += m * n;
  hist += m * 256;
  double* acc = reinterpret_cast<double*>(hist + 128);
  __shared__ unsigned int sh[100];
  for (int i = threadIdx.x; i < 100; i += blockDim.x) sh[i] = 0;
  __syncthreads();
  double nll = 0.0, se = 0.0, s2 = 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float sd = std[i], d = pred[i] - y[i];
    const float var = fmaxf(sd * sd, 1e-6f);
    nll += 0.5 * ((double)logf(var) + (double)d * d / var);
    se += (double)d * d;
    s2 += (double)sd * sd;
    // interval coverage: |z| <= icdf(0.5 + p/2)  <=>  erf(|z|/sqrt2) <= p ; first bin j with p_j >= q
    const float q = erff(fabsf(d / sd) * 0.70710678f);
    int j = (int)ceilf(q * 99.0f - 1e-6f);
    j = max(0, min(99, j));
    atomicAdd(&sh[j], 1u);
  }
  nll = block_sum(nll);
  se = block_sum(se);
  s2 = block_sum(s2);
  if (threadIdx.x == 0) { atomicAdd(acc + 0, nll); atomicAdd(acc + 1, se); atomicAdd(acc + 2, s2); }
  __syncthreads();
  for (int i = threadIdx.x; i < 100; i += blockDim.x)
    if (sh[i]) atomicAdd(hist + i, sh[i]);
}
__global__ void test_metrics_final_kernel(const unsigned int* hist, long long n, double* scalars, int nscal) {  // member = blockIdx.x
  if (threadIdx.x != 0) return;
  hist += blockIdx.x * 256ll;
  scalars += blockIdx.x * (long long)nscal;
  const double* acc = reinterpret_cast<const double*>(hist + 128);
  scalars[0] = acc[0] / (double)n;
  scalars[1] = acc[1] / (double)n;
  scalars[2] = sqrt(acc[2] / (double)n);
  double cum = 0.0, sq = 0.0, ab = 0.0;
  for (int j = 0; j < 100; ++j) {
    cum += hist[j];
    const double e = (double)j / 99.0 - cum / (double)n;
    sq += e * e;
    ab += fabs(e);
  }
  scalars[3] = sqrt(sq / 100.0);
  if (nscal > 4) scalars[4] = ab / 100.0;  // mean absolute calibration error (results/metrics.py:277-297)
}
void launch_test_metrics(const float* pred, const float* std, const float* y, long long n, double* scalars,
                         unsigned int* hist, cudaStream_t st, int nscal, int members) {
  // workspace layout, 1024 bytes per member: hist[100] u32 followed (at +512 B) by acc[3] doubles
  cudaMemsetAsync(hist, 0, (size_t)(members - 1) * 1024 + 512 + 3 * sizeof(double), st);
  ++g_launch_count;
  test_metrics_acc_kernel<<<dim3((unsigned)min((n + 255) / 256, (long long)148 * 4), (unsigned)members), 256, 0, st>>>(pred, std, y, n,
                                                                                                                   hist);
  ++g_launch_count;
  test_metrics_final_kernel<<<members, 32, 0, st>>>(hist, n, scalars, nscal);
}

// ------------------------------------------------------------------------------------------------
// ClippedAdam
// ------------------------------------------------------------------------------------------------
// The step size comes from the host (HostStep: brl_clipped_adam{,_vi}) or from a device table at a device index (DevStep: step k
// of brl_{elbo,hnn}_train_steps, whose launches are replayed from one graph)
struct HostStep {
  float v;
  __device__ __forceinline__ float get() const { return v; }
};
struct DevStep {
  const float* tab;
  const int* at;
  __device__ __forceinline__ float get() const { return tab[*at]; }
};
template <class Step>
__global__ void clipped_adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                    float* __restrict__ v, long long n, Step ss, float b1, float b2, float eps,
                                    float clip, float wd) {
  const float step_size = ss.get();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float gr = fminf(fmaxf(g[i], -clip), clip);
    const float pi = p[i];
    if (wd != 0.f) gr = fmaf(wd, pi, gr);
    const float mi = b1 * m[i] + (1.f - b1) * gr;
    const float vi = b2 * v[i] + (1.f - b2) * gr * gr;
    m[i] = mi;
    v[i] = vi;
    p[i] = pi - step_size * mi / (sqrtf(vi) + eps);
  }
}
// the optimiser step of a mean-field guide in one launch: ClippedAdam on loc and on log scale (the unconstrained parameter of
// Pyro's positive constraint), then scale = exp(log scale) for the next forward pass
template <class Step>
__global__ void clipped_adam_vi_kernel(float* __restrict__ loc, float* __restrict__ ls, float* __restrict__ scale,
                                       const float* __restrict__ g_loc, const float* __restrict__ g_ls, float* __restrict__ m_loc,
                                       float* __restrict__ v_loc, float* __restrict__ m_ls, float* __restrict__ v_ls, long long n,
                                       Step ss, float b1, float b2, float eps, float clip, float wd, float gscale) {
  const float step_size = ss.get();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    {
      float gr = fminf(fmaxf(g_loc[i] * gscale, -clip), clip);
      const float pi = loc[i];
      if (wd != 0.f) gr = fmaf(wd, pi, gr);
      const float mi = b1 * m_loc[i] + (1.f - b1) * gr, vi = b2 * v_loc[i] + (1.f - b2) * gr * gr;
      m_loc[i] = mi;
      v_loc[i] = vi;
      loc[i] = pi - step_size * mi / (sqrtf(vi) + eps);
    }
    {
      float gr = fminf(fmaxf(g_ls[i] * gscale, -clip), clip);
      const float pi = ls[i];
      if (wd != 0.f) gr = fmaf(wd, pi, gr);
      const float mi = b1 * m_ls[i] + (1.f - b1) * gr, vi = b2 * v_ls[i] + (1.f - b2) * gr * gr;
      m_ls[i] = mi;
      v_ls[i] = vi;
      const float pn = pi - step_size * mi / (sqrtf(vi) + eps);
      ls[i] = pn;
      scale[i] = expf(pn);
    }
  }
}
static DevStep dev_step(const TrainDesc* d) {  // device addresses of the descriptor's table and index
  const char* base = reinterpret_cast<const char*>(d);
  return DevStep{reinterpret_cast<const float*>(base + offsetof(TrainDesc, steps)), reinterpret_cast<const int*>(base + offsetof(TrainDesc, kt))};
}
template <class Step>
static void clipped_adam_vi_on(float* loc, float* ls, float* scale, const float* g_loc, const float* g_ls, float* m_loc, float* v_loc,
                               float* m_ls, float* v_ls, long long n, Step ss, float b1, float b2, float eps, float clip, float wd,
                               cudaStream_t st, float gscale) {
  ++g_launch_count;
  clipped_adam_vi_kernel<<<(unsigned)min((n + 255) / 256, (long long)148 * 8), 256, 0, st>>>(loc, ls, scale, g_loc, g_ls, m_loc, v_loc,
                                                                                            m_ls, v_ls, n, ss, b1, b2, eps, clip, wd,
                                                                                            gscale);
}
template <class Step>
static void clipped_adam_on(float* p, const float* g, float* m, float* v, long long n, Step ss, float b1, float b2, float eps,
                            float clip, float wd, cudaStream_t st) {
  ++g_launch_count;
  clipped_adam_kernel<<<(unsigned)min((n + 255) / 256, (long long)148 * 8), 256, 0, st>>>(p, g, m, v, n, ss, b1, b2, eps, clip, wd);
}
void launch_clipped_adam_vi(float* loc, float* ls, float* scale, const float* g_loc, const float* g_ls, float* m_loc, float* v_loc,
                            float* m_ls, float* v_ls, long long n, float step_size, float b1, float b2, float eps, float clip, float wd,
                            cudaStream_t st, float gscale) {
  clipped_adam_vi_on(loc, ls, scale, g_loc, g_ls, m_loc, v_loc, m_ls, v_ls, n, HostStep{step_size}, b1, b2, eps, clip, wd, st, gscale);
}
void launch_clipped_adam(float* p, const float* g, float* m, float* v, long long n, float step_size, float b1,
                         float b2, float eps, float clip, float wd, cudaStream_t st) {
  clipped_adam_on(p, g, m, v, n, HostStep{step_size}, b1, b2, eps, clip, wd, st);
}
void launch_clipped_adam_vi(float* loc, float* ls, float* scale, const float* g_loc, const float* g_ls, float* m_loc, float* v_loc,
                            float* m_ls, float* v_ls, long long n, const TrainDesc* d, float b1, float b2, float eps, float clip,
                            float wd, cudaStream_t st) {
  clipped_adam_vi_on(loc, ls, scale, g_loc, g_ls, m_loc, v_loc, m_ls, v_ls, n, dev_step(d), b1, b2, eps, clip, wd, st, 1.0f);
}
void launch_clipped_adam(float* p, const float* g, float* m, float* v, long long n, const TrainDesc* d, float b1, float b2, float eps,
                         float clip, float wd, cudaStream_t st) {
  clipped_adam_on(p, g, m, v, n, dev_step(d), b1, b2, eps, clip, wd, st);
}

// ------------------------------------------------------------------------------------------------
// torch.optim.Adam
// ------------------------------------------------------------------------------------------------
// Per element, what torch.optim.Adam's single-tensor path (fp32, amsgrad = maximize = False) computes, one torch op per line, each
// written with round-to-nearest intrinsics so that no contraction spans two torch ops (measured against torch on a B200: moments
// bit-identical without weight decay, parameters within 5.3e-8 of their largest magnitude, as far as torch's foreach path lies):
//   grad.add(param, alpha=wd)              g = fma(wd, p, g)                       (L2 weight decay, only when wd != 0)
//   exp_avg.lerp_(grad, w1)                m = fma(w1, g - m, m)  (w1 < 0.5; else fma(-(g - m), 1 - w1, g), torch's lerp)
//   exp_avg_sq.mul_(b2).addcmul_(g, g, w2) v = fma(w2, g g, v b2)
//   exp_avg_sq.sqrt() / bc2_sqrt + eps     d = sqrt(v) (1 / bc2_sqrt) + eps        (a tensor over a host scalar multiplies by its
//                                                                                   reciprocal, rounded in float)
//   param.addcdiv_(m, d, -step_size)       p = fma(-step_size, m / d, p)
// The (step_size, bc2_sqrt) pair comes from the host (HostAdam: brl_adam) or from the K-step call's table at a device index
// (DevAdam: brl_hnn_train_steps_adam).
struct HostAdam {
  float ss, bc2;
  __device__ __forceinline__ float2 get() const { return make_float2(ss, bc2); }
};
struct DevAdam {
  const float *ss, *bc2;
  const int* at;
  __device__ __forceinline__ float2 get() const {
    const int k = *at;
    return make_float2(ss[k], bc2[k]);
  }
};
template <class Step>
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                            long long n, Step sp, AdamArgs a) {
  const float2 s = sp.get();
  const float neg_ss = -s.x, inv_bc2 = __fdiv_rn(1.f, s.y);
  const bool small = fabsf(a.w1) < 0.5f;
  const float omw1 = __fsub_rn(1.f, a.w1);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float pi = p[i], mo = m[i], vo = v[i];
    float gr = g[i];
    if (a.wd != 0.f) gr = __fmaf_rn(a.wd, pi, gr);
    const float diff = __fsub_rn(gr, mo);
    const float mi = small ? __fmaf_rn(a.w1, diff, mo) : __fmaf_rn(-diff, omw1, gr);
    const float vi = __fmaf_rn(a.w2, __fmul_rn(gr, gr), __fmul_rn(vo, a.b2));
    const float den = __fadd_rn(__fmul_rn(__fsqrt_rn(vi), inv_bc2), a.eps);
    m[i] = mi;
    v[i] = vi;
    p[i] = __fmaf_rn(neg_ss, __fdiv_rn(mi, den), pi);
  }
}
template <class Step>
static void adam_on(float* p, const float* g, float* m, float* v, long long n, Step sp, const AdamArgs& a, cudaStream_t st) {
  ++g_launch_count;
  adam_kernel<<<(unsigned)min((n + 255) / 256, (long long)148 * 8), 256, 0, st>>>(p, g, m, v, n, sp, a);
}
void launch_adam(float* p, const float* g, float* m, float* v, long long n, float step_size, float bc2_sqrt, const AdamArgs& a,
                 cudaStream_t st) {
  adam_on(p, g, m, v, n, HostAdam{step_size, bc2_sqrt}, a, st);
}
void launch_adam(float* p, const float* g, float* m, float* v, long long n, const TrainDesc* d, const float* bc2, const AdamArgs& a,
                 cudaStream_t st) {
  const DevStep s = dev_step(d);
  adam_on(p, g, m, v, n, DevAdam{s.tab, bc2, s.at}, a, st);
}

// ------------------------------------------------------------------------------------------------
// K training steps per call (brl_elbo_train_steps / brl_hnn_train_steps): every per-step quantity is read from the call's
// descriptor in device memory, so one captured step serves every step of every later call with the same configuration
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void train_setup(const TrainSetup& s) {
  TrainDesc* d = s.d;
  for (int i = threadIdx.x; i < s.n; i += blockDim.x) d->steps[i] = s.steps[i];
  if (threadIdx.x == 0) {
    d->X = s.X; d->Y = s.Y; d->idx = s.idx; d->scalars = s.scalars; d->metrics = s.metrics;
    d->N = s.N; d->k = s.k0; d->kt = 0; d->bad = 0;
    d->seed = s.seed; d->sample0 = s.sample0; d->window0 = s.window0;
  }
}
__global__ void train_setup_kernel(const TrainSetup s) { train_setup(s); }
void launch_train_setup(const TrainSetup& s, cudaStream_t st) {
  ++g_launch_count;
  train_setup_kernel<<<1, 256, 0, st>>>(s);
}
// the same, plus torch Adam's sqrt(1 - beta2^t) column of this table
__global__ void train_setup_adam_kernel(const TrainSetupAdam s) {
  train_setup(s.s);
  for (int i = threadIdx.x; i < s.s.n; i += blockDim.x) s.bc2[i] = s.bc2_tab[i];
}
void launch_train_setup(const TrainSetupAdam& s, cudaStream_t st) {
  ++g_launch_count;
  train_setup_adam_kernel<<<1, 256, 0, st>>>(s);
}

// windows X[idx[k, w]] -> xb [MB,30,18] as float4 (a window is 135 of them), labels -> yb [MB]; an index outside [0, N) reads
// nothing (zeros) and marks the step; thread 0 writes step k's Philox key {seed + 0x9E3779B97F4A7C15 (k + 1), sample0, window0}
__global__ void train_gather_kernel(TrainDesc* d, float* __restrict__ xb, float* __restrict__ yb, long long MB) {
  const long long k = d->k, N = d->N;
  const long long* row = d->idx + k * MB;
  const float4* X = reinterpret_cast<const float4*>(d->X);
  const float* Y = d->Y;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < MB * 135; i += stride) {
    const long long w = i / 135, e = i - w * 135, j = row[w];
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (j >= 0 && j < N) v = __ldg(X + j * 135 + e);
    else if (e == 0) d->bad = 1;
    reinterpret_cast<float4*>(xb)[i] = v;
  }
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < MB; i += stride) {
    const long long j = row[i];
    yb[i] = (j >= 0 && j < N) ? __ldg(Y + j) : 0.f;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    d->dyn[0] = d->seed + 0x9E3779B97F4A7C15ull * (unsigned long long)(k + 1);
    d->dyn[1] = d->sample0;
    d->dyn[2] = d->window0;
  }
}
void launch_train_gather(TrainDesc* d, float* xb, float* yb, long long MB, cudaStream_t st) {
  ++g_launch_count;
  train_gather_kernel<<<(unsigned)min((MB * 135 + 255) / 256, (long long)148 * 8), 256, 0, st>>>(d, xb, yb, MB);
}

// member m's (loc, scale) pairs at src + m mstride -> the [M,B] planes of the step metrics
__global__ void split_pred_kernel(const float* __restrict__ src, long long mstride, long long B, float* pred, float* std) {
  const long long m = blockIdx.y;
  for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
    const float2 o = *reinterpret_cast<const float2*>(src + m * mstride + 2 * b);
    pred[m * B + b] = o.x;
    std[m * B + b] = o.y;
  }
}
void launch_split_pred(const float* src, long long mstride, int M, long long B, float* pred, float* std, cudaStream_t st) {
  ++g_launch_count;
  split_pred_kernel<<<dim3((unsigned)min((B + 255) / 256, (long long)148), (unsigned)M), 256, 0, st>>>(src, mstride, B, pred, std);
}

// the step's scalars [M,nscal] and metrics [M,5] -> row k of the caller's [K,M,.] buffers (NaN where the gather met a bad index);
// then the next step
__global__ void train_tail_kernel(TrainDesc* d, const double* __restrict__ scal, int nscal, const double* __restrict__ met, int M) {
  const long long k = d->k;
  const bool bad = d->bad != 0;
  const double nan = __longlong_as_double(0x7ff8000000000000ll);
  for (int i = threadIdx.x; i < M * nscal; i += blockDim.x) d->scalars[k * M * nscal + i] = bad ? nan : scal[i];
  for (int i = threadIdx.x; i < M * 5; i += blockDim.x) d->metrics[k * M * 5 + i] = bad ? nan : met[i];
  __syncthreads();
  if (threadIdx.x == 0) {
    d->k = k + 1;
    d->kt += 1;
    d->bad = 0;
  }
}
void launch_train_tail(TrainDesc* d, const double* scal, int nscal, const double* met, int M, cudaStream_t st) {
  ++g_launch_count;
  train_tail_kernel<<<1, 128, 0, st>>>(d, scal, nscal, met, M);
}

}  // namespace brl
