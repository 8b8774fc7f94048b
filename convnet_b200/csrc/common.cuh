// common.cuh — library-wide state and helpers (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "../../include/cudamat_abi.h"

namespace cnb {

// ---- error handling: same contract as the reference (cudamat_conv_gemm.cu:35-42):
// CUDA errors print and exit(EXIT_FAILURE); shape errors print and abort().
#define CNB_CUDA_CHECK(expr)                                                              \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      fprintf(stderr, "%s(%d) : convnet_b200 CUDA error : %s : (%d) %s.\n", __FILE__,     \
              __LINE__, #expr, (int)_e, cudaGetErrorString(_e));                          \
      exit(EXIT_FAILURE);                                                                 \
    }                                                                                     \
  } while (0)

#define CNB_LAUNCH_CHECK(what)                                                            \
  do {                                                                                    \
    cudaError_t _e = cudaGetLastError();                                                  \
    if (_e != cudaSuccess) {                                                              \
      fprintf(stderr, "%s(%d) : getLastCudaError() CUDA error : %s : (%d) %s.\n",         \
              __FILE__, __LINE__, what, (int)_e, cudaGetErrorString(_e));                 \
      exit(EXIT_FAILURE);                                                                 \
    }                                                                                     \
  } while (0)

#define CNB_REQUIRE(cond, what)                                                           \
  do {                                                                                    \
    if (!(cond)) {                                                                        \
      fprintf(stderr, "convnet_b200: %s: requirement failed: %s (%s:%d)\n", what, #cond,  \
              __FILE__, __LINE__);                                                        \
      abort();                                                                            \
    }                                                                                     \
  } while (0)

[[noreturn]] inline void not_implemented(const char* sym, const char* why) {
  fprintf(stderr, "convnet_b200: %s is not implemented: %s\n", sym, why);
  abort();
}

// programmatic dependent launch: this CTA does not mind the NEXT kernel of the stream being placed on the machine already
// (only kernels launched with the PDL attribute use it, and those wait for this grid's completion before their first
// global access — conv_tc.cu: launch_fast); a no-op for every other successor
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
// ... and the other half: block until every kernel this one depends on has completed and its writes are visible.  First
// statement of every kernel that launch_pdl() starts; a no-op when the launch carried no programmatic dependency.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// the dropout generator: a counter-based hash (splitmix64 finaliser) of seed + element index, top 32 bits -> [0, 1)
__host__ __device__ __forceinline__ uint32_t hash_u32(unsigned long long x) {
  x += 0x9E3779B97F4A7C15ULL; x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL; x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
  return (uint32_t)((x ^ (x >> 31)) >> 32);
}
__host__ __device__ __forceinline__ float dropout_keep(unsigned long long x, float dropprob, float scale) {
  return hash_u32(x) * (1.0f / 4294967296.0f) >= dropprob ? scale : 0.f;
}

// launch with programmatic stream serialization allowed (CONVNET_B200_NO_PDL=1: plain launch).  ONLY for kernels that
// execute pdl_wait() before their first global access.
inline bool pdl_enabled() {
  static const bool on = !(getenv("CONVNET_B200_NO_PDL") && getenv("CONVNET_B200_NO_PDL")[0] == '1');
  return on;
}
template <typename... KArgs, typename... Args>
inline void launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl_enabled() ? 1 : 0;
  CNB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...));
}

// ---- global state (one host thread per process/GPU, like the reference) -------------
enum Precision { kPrecFP32 = 0, kPrecTF32 = 1, kPrecBF16 = 2 };
enum ConvPath { kPathNone = -1, kPathSimt = 0, kPathTcTf32 = 1, kPathTcBf16 = 2 };
// which tensor-core kernel variant the last conv call ran (convnet_b200_last_conv_kernel); 0 for the CUDA-core path
enum ConvKernelBits {
  kKernLean = 1,              // tc_fast_kernel (else the general tc_conv_kernel)
  kKernPair = 2,              // CTA-pair mode (in any launch of the call)
  kKernXMode = 4,             // taps in the K block (Cin < 8)
  kKernSplit = 8,             // K split (fprop / dgrad + reduce_split) or reduction split (wgrad + reduce_partials)
  kKernDgradAsFprop = 16,     // dgrad as stride-1 fprop per stride phase; bits 8.. hold the phase count
  kKernAMerged = 32,          // fprop / dgrad: merged (image-fastest) A tensor map
  kKernBMerged = 64,          // fprop / dgrad: merged B tensor map
};
constexpr int kKernPhaseShift = 8;

// one-shot epilogue fusion requested for the next conv / pool-undo call (convnet_b200_fuse_next)
struct Fuse {
  const float* bias = nullptr;       // fprop: + bias[output channel]
  int relu = 0;                      // fprop: max(., 0) after the bias
  const float* relu_mask = nullptr;  // dgrad / pool undo: result zeroed where relu_mask <= 0 (same shape as the target)
  // fprop: dropout after bias / ReLU (convnet_b200_fuse_next_dropout): element i (its index in the target tensor) is kept
  // iff dropout_uniform(seed + i) >= drop_prob, kept values are multiplied by drop_scale; drop_scale == 0: no dropout
  float drop_prob = 0.f, drop_scale = 0.f; unsigned long long drop_seed = 0;
  bool* dropped = nullptr;           // internal: the kernel sets it when it applied the dropout itself
  int prestage = 0;                  // convDown*: only build what the call can prepare from the FILTERS (convnet_b200_prestage_next)
  int pool_cache = 0;                // MaxPool*: also record the tie masks for the matching MaxPoolUndo* (convnet_b200_pool_cache_next)
  float out_scale = 1.f;             // dgrad: result multiplied by this (the kept-unit scale of a dropout layer, see ext.h)
  int emit_bf16 = 0;                 // any writer: also leave a staged bf16 copy of the whole target (convnet_b200_emit_bf16_next)
  // the writer also produces the bias gradient of the edge that consumes the target as its output derivative
  // (convnet_b200_fuse_next_bias_grad): grad_bias[c] = bg_st*grad_bias[c] + bg_so * sum over images and positions
  float* bias_grad = nullptr; float bg_st = 0.f, bg_so = 1.f;
  // internal (filled by the ABI wrapper): where the bf16 twin of the target goes; a kernel that writes it sets *emitted
  __nv_bfloat16* out16 = nullptr;
  bool* emitted = nullptr;
  bool any() const { return bias || relu || relu_mask || drop_scale != 0.f; }
};

struct State {
  cudaStream_t stream = 0;          // legacy default stream, like every reference kernel
  int precision = kPrecFP32;      // the raw C ABI computes in fp32 (the reference's arithmetic) until a caller opts into tf32 / bf16
  int last_conv_path = kPathNone;
  int last_conv_kernel = -1;        // ConvKernelBits of the same call
  unsigned long long launches = 0;  // kernels launched by this library
  // scratch (wgrad partial sums, rnorm-free) — grown on demand, never per-call malloc'd
  void* ws = nullptr;
  size_t ws_bytes = 0;
  int ws_device = -1;
  int num_sms = 0;
  int sm_device = -1;
  int sm_reserve = 0;                 // SMs the persistent conv grids leave free (convnet_b200_reserve_sms)
  Fuse fuse;
};
inline Fuse take_fuse();
State& state();

void* workspace(size_t bytes);       // device scratch of at least `bytes`, valid until next call
int num_sms();
inline int current_device() { int d = 0; CNB_CUDA_CHECK(cudaGetDevice(&d)); return d; }

inline void count_launch(int n = 1) { state().launches += n; }
inline void note_conv(int path, int kernel) { state().last_conv_path = path; state().last_conv_kernel = kernel; }
inline Fuse take_fuse() { Fuse f = state().fuse; state().fuse = Fuse(); return f; }

template <typename T>
__host__ __device__ inline T ceil_div(T a, T b) { return (a + b - 1) / b; }

}  // namespace cnb
