// ext.cu — library state, scratch, and the extension C API (include/convnet_b200_ext.h).
#include <string.h>

#include "../../include/convnet_b200_ext.h"
#include "common.cuh"
#include "conv_kernels.h"

namespace cnb {

State& state() {
  static State s;
  static bool init = false;
  if (!init) {
    init = true;
    const char* e = getenv("CONVNET_B200_PRECISION");
    if (e) {
      if (!strcmp(e, "fp32")) s.precision = kPrecFP32;
      else if (!strcmp(e, "tf32")) s.precision = kPrecTF32;
      else if (!strcmp(e, "bf16")) s.precision = kPrecBF16;
      else { fprintf(stderr, "convnet_b200: unknown CONVNET_B200_PRECISION '%s'\n", e); abort(); }
    }
  }
  return s;
}

void* workspace(size_t bytes) {
  State& s = state();
  int dev = 0;
  CNB_CUDA_CHECK(cudaGetDevice(&dev));
  if (s.ws && (s.ws_device != dev || s.ws_bytes < bytes)) {
    // growing: wait for users of the old block on our stream, then free
    CNB_CUDA_CHECK(cudaStreamSynchronize(s.stream));
    int cur = dev;
    if (s.ws_device != dev) CNB_CUDA_CHECK(cudaSetDevice(s.ws_device));
    CNB_CUDA_CHECK(cudaFree(s.ws));
    if (s.ws_device != cur) CNB_CUDA_CHECK(cudaSetDevice(cur));
    s.ws = nullptr; s.ws_bytes = 0;
  }
  if (!s.ws) {
    size_t want = bytes < (size_t(64) << 20) ? (size_t(64) << 20) : bytes;
    cudaError_t e = cudaMalloc(&s.ws, want);
    if (e != cudaSuccess) {
      fprintf(stderr, "convnet_b200: could not allocate %zu bytes of scratch: %s\n", want, cudaGetErrorString(e));
      exit(EXIT_FAILURE);
    }
    s.ws_bytes = want; s.ws_device = dev;
  }
  return s.ws;
}

int num_sms() {
  State& s = state();
  int dev = 0;
  CNB_CUDA_CHECK(cudaGetDevice(&dev));
  if (s.sm_device != dev) {
    CNB_CUDA_CHECK(cudaDeviceGetAttribute(&s.num_sms, cudaDevAttrMultiProcessorCount, dev));
    s.sm_device = dev;
  }
  const int usable = s.num_sms - s.sm_reserve;
  return usable >= 8 ? usable : (s.num_sms < 8 ? s.num_sms : 8);
}

}  // namespace cnb

using namespace cnb;

extern "C" {

int convnet_b200_version(void) { return 100; }
void convnet_b200_set_stream(void* cuda_stream) { state().stream = (cudaStream_t)cuda_stream; }
void* convnet_b200_get_stream(void) { return (void*)state().stream; }
void convnet_b200_set_conv_precision(int mode) {
  CNB_REQUIRE(mode >= 0 && mode <= 2, "convnet_b200_set_conv_precision");
  if (mode != state().precision) bf16_invalidate(nullptr);      // staged copies do not survive a mode change
  state().precision = mode;
}
int convnet_b200_get_conv_precision(void) { return state().precision; }
void convnet_b200_fuse_next(const float* bias, int relu, const float* relu_mask) {
  state().fuse.bias = bias; state().fuse.relu = relu; state().fuse.relu_mask = relu_mask;
}
void convnet_b200_emit_bf16_next(void) { state().fuse.emit_bf16 = 1; }
void convnet_b200_fuse_next_bias_grad(float* grad_bias, float scaleTargets, float scaleOutput) {
  state().fuse.bias_grad = grad_bias; state().fuse.bg_st = scaleTargets; state().fuse.bg_so = scaleOutput;
}
void convnet_b200_fuse_next_scale(float scale) { state().fuse.out_scale = scale; }
void convnet_b200_pool_cache_next(void) { state().fuse.pool_cache = 1; }
void convnet_b200_prestage_next(void) { state().fuse.prestage = 1; }
int convnet_b200_extract_patches(cudamat* images, cudamat* patches, cudamat* width_offset, cudamat* height_offset,
                                 cudamat* flip, int img_width, int img_height, int patch_width, int patch_height) {
  // argument checks of cudamat.cu:2699-2713
  if (img_width <= 0 || img_height <= 0 || patch_width <= 0 || patch_height <= 0) return -1;
  const int num_images = images->size[1];
  const int num_colors = images->size[0] / (img_width * img_height);
  if (num_colors <= 0 || images->size[0] != num_colors * img_width * img_height) return -1;
  if (patches->size[1] != num_colors * patch_width * patch_height || patches->size[0] != num_images) return -1;
  if (width_offset->size[0] * width_offset->size[1] != num_images) return -1;
  if (height_offset->size[0] * height_offset->size[1] != num_images) return -1;
  if (flip->size[0] * flip->size[1] != num_images) return -1;
  return extract_patches(images->data_device, patches->data_device, width_offset->data_device, height_offset->data_device,
                         flip->data_device, num_images, img_width, img_height, patch_width, patch_height, num_colors);
}
void convnet_b200_fuse_next_dropout(float dropprob, float scale, unsigned long long seed) {
  Fuse& f = state().fuse;
  f.drop_prob = dropprob; f.drop_scale = scale; f.drop_seed = seed;
}
void convnet_b200_reserve_sms(int n) { state().sm_reserve = n > 0 ? n : 0; }
void convnet_b200_bf16_stage(const float* ptr, long long n) { bf16_stage(ptr, n); }
void convnet_b200_bf16_ensure(const float* ptr, long long n) { bf16_ensure(ptr, n); }
int convnet_b200_bf16_is_staged(const float* ptr, long long n) { return want_bf16() && bf16_staged(ptr, n) != nullptr; }
void convnet_b200_bf16_invalidate(const float* ptr) { bf16_invalidate(ptr); }
int convnet_b200_last_conv_path(void) { return state().last_conv_path; }
int convnet_b200_last_conv_kernel(void) { return state().last_conv_kernel; }
unsigned long long convnet_b200_launch_count(void) { return state().launches; }
void convnet_b200_reset_launch_count(void) { state().launches = 0; }
void convnet_b200_release_workspace(void) {
  State& s = state();
  bf16_release();
  if (s.ws) {
    CNB_CUDA_CHECK(cudaStreamSynchronize(s.stream));
    CNB_CUDA_CHECK(cudaFree(s.ws));
    s.ws = nullptr; s.ws_bytes = 0; s.ws_device = -1;
  }
}

}  // extern "C"
