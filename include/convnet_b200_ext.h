/* convnet_b200_ext.h — additions to the reference's C surface (everything here is
 * new; nothing replaces a reference symbol).  Plain C ABI: pointers and scalars only.
 */
#ifndef CONVNET_B200_EXT_H_
#define CONVNET_B200_EXT_H_

#include "cudamat_abi.h"

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)   /* the library is built with -fvisibility=hidden */
#endif

/* Library version (major*10000 + minor*100 + patch). */
int convnet_b200_version(void);

/* Stream every kernel of this library is enqueued on.  Default: the legacy
 * default stream 0, which is what every reference kernel uses
 * (cudamat_conv_filteracts.cu:1259), so ordering against libcudamat.so is kept.
 * `cuda_stream` is a cudaStream_t / CUstream handle. */
void convnet_b200_set_stream(void* cuda_stream);
void* convnet_b200_get_stream(void);

/* Arithmetic of the three conv ops (pool / response-norm are always fp32):
 *   0  FP32  fp32 FMA on CUDA cores (the DEFAULT: a drop-in caller gets the reference's arithmetic); meets the
 *            reference's own 1e-4 kernel test tolerance (py/test_conv.py:387); what run_grad_check uses
 *   1  TF32  tcgen05 kind::tf32 on the caller's fp32 buffers, fp32 accumulate;
 *            Diff <= 5e-3 (operands truncated to 10 mantissa bits by the tensor core)
 *   2  BF16  tcgen05 kind::f16 on bf16 copies, fp32 accumulate; Diff <= 2e-2
 * Shapes the tensor-core path does not take fall through to FP32.  The tensor-core modes are opt-in: this call, or
 * CONVNET_B200_PRECISION={fp32,tf32,bf16} in the environment before first use (host/ConvNet and bench.py opt in). */
void convnet_b200_set_conv_precision(int mode);
int convnet_b200_get_conv_precision(void);

/* Which path the most recent conv call took: 0 CUDA-core fp32, 1 tcgen05 tf32,
 * 2 tcgen05 bf16, -1 none yet.  (tests assert the tensor path really ran) */
int convnet_b200_last_conv_path(void);

/* Which kernel variant the most recent conv call ran, as a bit mask (0 for the CUDA-core path, -1 none yet).  It only
 * records what the shape and the mode selected; tests use it to prove a case reaches the variant it exists for.
 *   1 lean kernel          2 CTA pair (in any launch of the call)      4 x-mode (Cin < 8: filter taps in the K block)
 *   8 K split (fprop / dgrad) or reduction split (wgrad) > 1           16 dgrad run as stride-1 fprop per stride phase
 *   32 merged A tensor map (fprop / dgrad)                             64 merged B tensor map (fprop / dgrad)
 *   bits 8..12: number of stride phases of a dgrad-as-fprop call */
int convnet_b200_last_conv_kernel(void);

/* Number of kernels this library has launched since the last reset. */
unsigned long long convnet_b200_launch_count(void);
void convnet_b200_reset_launch_count(void);

/* One-shot: the NEXT pool-undo (MaxPoolUndo*, AvgPoolUndo*) or convDown* call also produces the shared-bias gradient of
 * the edge BELOW — the one whose output derivative is the tensor this call writes (src/conv_edge.cc:210-222 runs
 * SumRows over that tensor later):  grad_bias[c] = scaleTargets*grad_bias[c] + scaleOutput * sum_{n,pixels} target[n,pixel,c].
 * The sums come from the values the kernel is storing anyway (deterministic per-row partial sums + a tiny second
 * kernel), so the separate pass over the derivative disappears; calls that cannot do it run that pass themselves. */
void convnet_b200_fuse_next_bias_grad(float* grad_bias, float scaleTargets, float scaleOutput);

/* One-shot: the NEXT convDown* call multiplies its result by `scale` (before the relu_mask of convnet_b200_fuse_next).
 * This is how the derivative of inverted dropout disappears as a pass: for a ReLU layer with dropout the state holds
 * relu(x) * m with m in {0, 1/(1-p)}, so  deriv * m * [state > 0]  (Layer::ApplyDerivativeofDropout followed by
 * ApplyDerivativeOfActivation, src/layer.cc:367-395,562-580)  ==  deriv * 1/(1-p) * [state > 0]. */
void convnet_b200_fuse_next_scale(float scale);

/* One-shot: the NEXT MaxPool* call also records which elements of every window equal its maximum (one 16-bit mask per
 * pooled element, in library scratch).  The MaxPoolUndo* call on the same (images, maxActs) pair then reads the gradients
 * and those masks instead of re-reading the pool input and output and comparing — 0.55x the bytes of the largest
 * memory-bound pass of the step, bit-identical results (ties duplicate the gradient exactly as kMaxPoolUndo's `==` test
 * does, cudamat_conv_gemm.cu:262-300).  The masks go stale, and the undo falls back to comparing, as soon as any entry
 * point of this library writes either tensor; a caller that overwrites them by other means between the two calls must
 * not use this request (or must call convnet_b200_bf16_invalidate(NULL)).  2-D windows up to 3 x 3. */
void convnet_b200_pool_cache_next(void);

/* One-shot request for the next convUp* call (after its bias / ReLU, if those are requested too): dropout of the result with
 * the generator of cnb_dropout — element i of the target is kept iff hash(seed + i) >= dropprob, kept values are multiplied
 * by `scale` — exactly as if cnb_dropout(target, mask, n, dropprob, scale, seed) followed the call, except that NO mask
 * tensor is written: the caller's backward pass must not need one (for a ReLU layer the kept units are the non-zero ones:
 * convnet_b200_fuse_next_scale on the dgrad that produces this layer's derivative).  The bf16 lean kernels apply it in
 * the epilogue; every other path runs one trailing pass inside the call. */
void convnet_b200_fuse_next_dropout(float dropprob, float scale, unsigned long long seed);

/* One-shot request for the next convDown* call: do not compute anything, only prepare on the current stream what that call
 * derives from the FILTERS alone — in bf16 mode the per-stride-phase, tap-flipped bf16 filter banks the dgrad kernels read
 * (DESIGN.md §3).  The derivative and target tensors are not touched (their shapes must still describe the call).  A
 * trainer issues this right after the optimizer step of a layer, on the optimizer's stream, so that the next step's
 * convDown finds the banks ready instead of rebuilding them on the critical path. */
void convnet_b200_prestage_next(void);

/* The conv kernels are persistent: one CTA (or CTA pair) per SM, each owning most of the SM's shared memory.  A kernel
 * of another library that must run CONCURRENTLY (an NCCL collective on a side stream) cannot co-reside with them and
 * would otherwise wait for — or push out — a whole wave.  convnet_b200_reserve_sms(n) makes the persistent grids leave
 * n SMs free until it is called again with 0.  (host/convnet.cc reserves the SMs of the gradient all-reduce while it
 * is in flight.) */
void convnet_b200_reserve_sms(int n);

/* Free cached device scratch (wgrad / split-K partial sums, bf16 staging buffers).  Never required. */
void convnet_b200_release_workspace(void);

/* One-shot epilogue fusion for the NEXT conv / pool-undo call of this library (cleared by that call):
 *   bias      (convUp*, localUp excluded): adds bias[o] to every output of output channel o — the shared-bias
 *             AddRowVec of ConvEdge::ComputeUp (src/conv_edge.cc:143-152) without the extra pass;
 *   relu      (convUp*): clamps at 0 after the bias — Layer::ApplyActivation for RECTIFIED_LINEAR (src/layer.cc:550);
 *   relu_mask (convDown*, MaxPoolUndo*, AvgPoolUndo*): result zeroed where relu_mask[i] <= 0; relu_mask has the shape
 *             of `targets` (it is the state of the layer receiving the derivative: ApplyDerivativeOfActivation).
 * Pass NULL / 0 for the parts not wanted.  Calls that cannot fuse (3-D dgrad) apply the same maths in a second pass. */
void convnet_b200_fuse_next(const float* bias, int relu, const float* relu_mask);

/* bf16 operand staging (precision mode 2 only; no-ops in the other modes).  In bf16 mode every conv call first rounds
 * its two fp32 operands to bf16 copies.  A caller that knows a tensor stays unchanged across several conv calls
 * (the layer input: fprop + wgrad; the output derivative: wgrad + dgrad; the weights: fprop + dgrad) can have it
 * converted ONCE: convnet_b200_bf16_stage(ptr, n) converts the n floats at ptr now (stream-ordered) and conv calls
 * that receive exactly `ptr` as an operand use that copy while it is valid.  convnet_b200_bf16_ensure converts only
 * when no valid copy exists.
 * Coherence: every entry point of THIS library that writes a tensor drops the staged copies overlapping what it
 * writes (and convnet_b200_emit_bf16_next makes it leave a fresh one), and cnb_sgd_momentum refreshes the copy of
 * the weights it updates.  Only writes the library cannot see (cudaMemcpy, another library's kernels) need an
 * explicit convnet_b200_bf16_invalidate(ptr) / _stage(ptr, n) from the caller; convnet_b200_bf16_invalidate(NULL)
 * forgets every staged tensor.  CONVNET_B200_STAGE_VERIFY=1 (environment) re-converts the fp32 source at every use of
 * a staged copy and aborts on a mismatch — the way to find such a missed write. */
void convnet_b200_bf16_stage(const float* ptr, long long n);
void convnet_b200_bf16_ensure(const float* ptr, long long n);
void convnet_b200_bf16_invalidate(const float* ptr);
int convnet_b200_bf16_is_staged(const float* ptr, long long n);   /* 1 if a valid staged copy covers [ptr, ptr+n) */

/* One-shot: the NEXT entry point of this library that writes a tensor (conv fprop / dgrad, pooling and its undo,
 * response norm and its undo, cnb_relu, cnb_dropout, cnb_mult, cnb_add_channel_bias*) also leaves a staged bf16 copy of
 * the WHOLE target tensor, exactly as convnet_b200_bf16_stage(target, n) right after the call would — but written by the
 * producing kernel from the same registers where that kernel supports it (the fp32 -> bf16 pass and its 6 bytes/element
 * of HBM traffic disappear), by a trailing conversion pass where it does not.  No-op outside bf16 mode. */
void convnet_b200_emit_bf16_next(void);

/* ---- steps either side of the conv ops that the Edge layer sequences ------------
 * (SURVEY.md §8(f) rank 2; in the reference these are libcudamat.so calls:
 *  add_row_vec cudamat.cu:1064, sum_by_axis :1614, lower_bound_scalar :1426,
 *  apply_rectified_linear_deriv :2475).  Names are prefixed so both libraries link. */

/* acts (N, locs, C): acts[n, l, c] += bias[c]  — ConvEdge::ComputeUp shared bias,
 * src/conv_edge.cc:143-152.  rows = N*locs, cols = C. */
void cnb_add_channel_bias(float* acts, const float* bias, long long rows, int cols);
/* same, fused with ReLU (Layer::ApplyActivation, src/layer.cc:550: LowerBound(0)). */
void cnb_add_channel_bias_relu(float* acts, const float* bias, long long rows, int cols);
/* grad_bias[c] = scaleTargets*grad_bias[c] + scaleOutput * sum_{rows} derivs[r, c]
 * — src/conv_edge.cc:210-222 (two-step SumRows). Deterministic. */
void cnb_channel_bias_grad(const float* derivs, float* grad_bias, long long rows, int cols,
                           float scaleTargets, float scaleOutput);
/* x = max(x, 0) ; dx *= (y > 0) */
void cnb_relu(float* x, long long n);
void cnb_relu_deriv(float* dx, const float* y, long long n);
/* binary dropout (Layer::ApplyDropoutAtTrainTime, src/layer.cc:367-395): mask[i] = Bernoulli(1-dropprob)*scale,
 * x *= mask; counter-based RNG keyed by (seed, i).  cnb_mult: a *= b (ApplyDerivativeofDropout). */
void cnb_dropout(float* x, float* mask, long long n, float dropprob, float scale, unsigned long long seed);
void cnb_mult(float* a, const float* b, long long n);
/* softmax over the classes of a column-major [rows=N x cols=classes] matrix, in place
 * (Layer::ApplyActivation for SOFTMAX layers, src/layer.cc) */
void cnb_softmax(float* x, int rows, int cols);
/* deriv = probs - onehot(labels); loss_per_image[n] = -log probs[n, label] (may be NULL)
 * (CrossEntropyMultinomial, src/loss_functions.cc:70-95) */
void cnb_softmax_ce_deriv(const float* probs, const int* labels, float* deriv, float* loss_per_image,
                          int rows, int cols);
/* *out = sum(a[0..n)) on the device (no host sync) */
void cnb_sum(const float* a, float* out, int n);
/* SGD with momentum and L2 decay, one fused pass (src/optimizer.cc:174-200):
 *   g' = lr*(g + l2*w);  h = momentum*h + g';  w -= h */
void cnb_sgd_momentum(float* w, float* hist, const float* grad, long long n, float lr,
                      float momentum, float l2);
/* the same update for `count` tensors in ONE launch (one call per all-reduce bucket / per net instead of one per
 * weight and bias matrix).  `tensors` is a host array.  In bf16 mode a staged copy of a weight tensor is refreshed
 * by the same pass (see convnet_b200_bf16_stage). */
typedef struct CnbSgdTensor {
  float* w; float* hist; const float* grad; long long n; float lr, momentum, l2;
} CnbSgdTensor;
void cnb_sgd_momentum_multi(const CnbSgdTensor* tensors, int count);

/* ---- input pipeline, device side (SURVEY.md §8 f4) -------------------------------------------------------------------
 * The reference keeps a chunk of the data set on the GPU, one image per COLUMN (pixel index = col + W*(row + H*color)),
 * and cuts every minibatch out of it with a random crop and mirror per image while transposing it into the image-fastest
 * layout of the input layer: DataIterator::AddNoise -> Matrix::ExtractPatches (src/datahandler.cc:520-531,
 * src/matrix.cc:1030-1042) -> extract_patches (cudamat/cudamat.cuh:265, cudamat.cu:2699-2742, kernel
 * cudamat_kernels.cu:1655-1669).  Same arguments, same element-for-element result, same error codes
 * (ERROR_INCOMPATIBLE_DIMENSIONS = -1, CUDA_ERROR = -3); exported under its own name because the reference's copy lives in
 * libcudamat.so, which a drop-in build keeps linking:
 *   patches[n + N*(x + pw*(y + ph*c))] = images[sx + W*(height_offset[n] + y + H*(c + C*n))],
 *   sx = width_offset[n] + x, mirrored to W - 1 - sx when flip[n] > 0.5.
 * `images` is (C*W*H) x N in cudamat's size[] convention (size[1] = N images), `patches` is N x (C*pw*ph); the three
 * per-image vectors hold N floats on the device.  Source coordinates are clamped to the image (the reference reads out of
 * bounds for a crop that does not fit).  Runs on the library's stream. */
int convnet_b200_extract_patches(cudamat* images, cudamat* patches, cudamat* width_offset, cudamat* height_offset,
                                 cudamat* flip, int img_width, int img_height, int patch_width, int patch_height);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif  /* CONVNET_B200_EXT_H_ */
