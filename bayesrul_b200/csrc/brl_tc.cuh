// tcgen05 / TMEM engine (fp16 operands, fp32 accumulate) -- interface used by brl_api.cu.
#pragma once
#include <cstddef>
#include <cuda_runtime.h>

struct brl_noise;

namespace brl {
struct TcState;
TcState* tc_create(int net);
void tc_destroy(TcState*);
bool tc_available(const TcState*);      // Inception: fused conv + fc kernels; Linear: brl_tc_linear.cuh
bool tc_host_pipeline(const TcState*);  // chunked host-batch pipeline with prepacked weight images (Inception only)
int tc_status(const TcState*);  // 0 ok; else the code of the first mbarrier wait that timed out (synchronises)
void tc_timing(TcState*, bool enable);
void tc_timing_read(TcState*, double ms[2], long long launches[2]);  // [conv, fc]; synchronises the recorded events
void tc_trace(TcState*, long long* device_buf);
// false while brl_tc_timing brackets launches with events or brl_tc_trace names a buffer: those host-side hooks act at enqueue
// time, so a captured forward would replay without them (and with a trace pointer that may be gone); run such forwards eagerly
bool tc_capturable(const TcState*);
size_t tc_workspace_bytes(const TcState*, long long B, long long S);
// returns nullptr on success, else a static error string.  pack_x = false re-uses the fp16 window images a previous
// call built in the same workspace for the same x (later chunks of MC samples of one batch).
// prepacked != nullptr: the fp16 weight images of the S samples (tc_pack_weights) are taken from there instead of being
// packed from `weights` into the workspace (window chunks of one batch share the images of all MC samples).
// With w_sample_stride != 0, MC sample s uses weight row / image (s + img_phase) / img_per: img_per = 1 is one image per sample;
// img_per = S serves the samples of several ensemble members (S each, the first member img_phase samples in) from one image per
// member.  w_sample_stride == 0: one image shared by all samples.
const char* tc_forward(TcState*, const float* x, long long B, long long S, const float* weights, long long w_sample_stride,
                       float p_dropout, const brl_noise* noise, float* out, void* ws, size_t ws_bytes, bool pack_x,
                       cudaStream_t st, const unsigned char* prepacked = nullptr, int img_per = 1, int img_phase = 0);
size_t tc_weight_image_bytes();  // bytes of one sample's fp16 weight image
// fp32 weights [n, P] (or one shared [P] vector: n = 1) -> n fp16 weight images at `images` (tc_weight_image_bytes() apart).
// The images depend on p_dropout (inverted dropout's 1 / keep is folded into the weights behind a dropout site): pass the value
// the images will be used with in tc_forward.
const char* tc_pack_weights(TcState*, const float* weights, long long w_sample_stride, long long n, unsigned char* images,
                            float p_dropout, cudaStream_t st);
}  // namespace brl
