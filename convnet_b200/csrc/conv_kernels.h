// conv_kernels.h — host-side entry points of the kernel translation units.
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"
#include "geom.h"

namespace cnb {

// conv_simt.cu — fp32 CUDA-core implicit GEMM (exact mode + shapes the tensor path skips)
void simt_conv_up(const ConvGeom& g, const float* images, const float* filters, float* targets,
                  float scaleTargets, float scaleOutput, const Fuse& fuse);
void simt_conv_down(const ConvGeom& g, const float* derivs, const float* filters, float* targets,
                    float scaleTargets, float scaleOutput, const Fuse& fuse);
// rectH x rectW: module rectangle per reduction chunk; keep_partials: one output block per chunk
void simt_conv_outp(const ConvGeom& g, const float* images, const float* derivs, float* targets,
                    int rectH, int rectW, bool keep_partials, float scaleTargets, float scaleOutput);
void scale_buffer(float* a, long long n, float s);
void reduce_partials(const float* part, float* out, long long elems, int groups, int per, float st, float so);

// conv_tc.cu — tcgen05 / TMA implicit GEMM (sm_100a tensor cores)
bool tc_conv_up(const ConvGeom& g, const float* images, const float* filters, float* targets,
                float scaleTargets, float scaleOutput, const Fuse& fuse);
int extract_patches(const float* images, float* patches, const float* width_offset, const float* height_offset, const float* flip,
                    int N, int W, int H, int pw, int ph, int C);                                          // elementwise.cu
void dropout_apply(float* x, long long n, float dropprob, float scale, unsigned long long seed, __nv_bfloat16* out16);   // elementwise.cu
void tc_conv_down_prestage(const ConvGeom& g, const float* derivs, const float* filters);   // builds the dgrad filter banks, if that path will run
bool tc_conv_down(const ConvGeom& g, const float* derivs, const float* filters, float* targets,
                  float scaleTargets, float scaleOutput, const Fuse& fuse);
bool tc_conv_outp(const ConvGeom& g, const float* images, const float* derivs, float* targets,
                  float scaleTargets, float scaleOutput);

// stage.cu — bf16 operand copies and their coherence (convnet_b200_bf16_stage / _ensure / _invalidate / emit)
bool want_bf16();
void to_bf16(const float* src, __nv_bfloat16* dst, long long n);
const __nv_bfloat16* bf16_staged(const float* src, long long n);      // valid copy covering [src, src+n), or nullptr
void bf16_stage(const float* ptr, long long n);                        // convert now
void bf16_ensure(const float* ptr, long long n);                       // convert unless a valid copy exists
void bf16_invalidate(const float* ptr);
void bf16_note_write(const float* ptr, long long n);                   // [ptr, ptr+n) is being overwritten: overlapping copies go stale
__nv_bfloat16* bf16_emit_slot(const float* ptr, long long n);          // buffer a producing kernel fills itself (marked valid)
__nv_bfloat16* bf16_refresh_slot(const float* ptr, long long n);       // the existing buffer of exactly this tensor, or nullptr
void bf16_release();                                                   // drops the buffers too
// dgrad in fprop form (stage.cu): stride phases and the per-phase filter banks [c][tap''][o]
constexpr int kMaxDgradPhases = 16;
struct DgradPhase {
  int a, b;            // input pixel phase: x = sx*i + a, y = sy*j + b
  int rx, ry;          // tap residues: tx = rx + sx*u
  int ku, kv;          // taps of this phase
  int px, py;          // (negative) window start offsets of the stride-1 correlation over the derivative
  int Wp, Hp;          // pixels of this phase
  long long offset;    // element offset of the phase's bank
};
struct DgradBanks { int count; DgradPhase phase[kMaxDgradPhases]; };
int dgrad_phases(const ConvGeom& g, DgradBanks* b);                    // number of phases, or -1 if there are too many
// the banks of `filters`: cached ones when valid, else built now; `keep`: they stay cached (prestage), else they serve this call only
const __nv_bfloat16* dgrad_weights(const float* filters, const ConvGeom& g, const DgradBanks& b, bool keep);
// max-pool tie masks (stage.cu), see pool.cu
uint16_t* pool_masks_slot(const float* acts, long long n_out, const float* images, long long n_in, unsigned long long sig);
const uint16_t* pool_masks_find(const float* acts, long long n_out, const float* images, unsigned long long sig);
// writer protocol: begin_write drops stale copies and returns the buffer the kernel must fill when it can emit; end_write
// falls back to a conversion pass when emission was wanted but the kernel could not do it
__nv_bfloat16* begin_write(float* target, long long n, bool want_emit, bool kernel_can_emit);
void end_write(float* target, long long n, bool want_emit, const __nv_bfloat16* emitted);

// pool.cu
// targets_bf16 (may be null): also write the bf16 twin of the target; the return value says whether the kernel did
bool pool_forward(const PoolGeom& g, bool is_max, const float* images, float* targets, float scaleOutput,
                  __nv_bfloat16* targets_bf16 = nullptr, bool cache_masks = false);
// colsum / colsum_slices (may be null): where a kernel that can do so leaves per-slice channel sums of the tensor it wrote,
// colsum[slice * channels + c] (*colsum_slices = number of slices, 0 = not done) — the bias gradient of the edge below
bool max_pool_undo(const PoolGeom& g, const float* images, const float* maxGrads, const float* maxActs,
                   float* targets, float scaleTargets, float scaleOutput, const float* relu_mask,
                   __nv_bfloat16* targets_bf16 = nullptr, float* colsum = nullptr, int* colsum_slices = nullptr);
bool avg_pool_undo(const PoolGeom& g, const float* avgGrads, float* targets, float scaleTargets,
                   float scaleOutput, const float* relu_mask, __nv_bfloat16* targets_bf16 = nullptr,
                   float* colsum = nullptr, int* colsum_slices = nullptr);
// grad_bias[c] = st*grad_bias[c] + so * sum_slices part[slice*cols + c]   (elementwise.cu)
void colsum_finish(const float* part, float* grad_bias, int cols, int slices, float st, float so);

// rnorm.cu
// relu / targets_bf16: fused epilogue (max(., 0); a bf16 copy of the output) — only when rnorm_can_fuse(numFilters)
void rnorm_forward(const float* images, float* targets, long long num_locs, int numFilters, int sizeF,
                   float addScale, float powScale, bool blocked, bool relu = false, __nv_bfloat16* targets_bf16 = nullptr);
bool rnorm_can_fuse(int numFilters);
void rnorm_undo(const float* outGrads, const float* inputs, float* targets, long long num_locs,
                int numFilters, int sizeF, float addScale, float powScale, bool blocked);

}  // namespace cnb
