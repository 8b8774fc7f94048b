// abi.cu — the extern "C" surface: ABI-1 (include/convnet_b200_conv_gemm.h, the
// reference's cudamat_conv_gemm.cuh) and ABI-2 (include/convnet_b200_conv.h, the
// reference's cudamat_conv.cuh), both on the same kernels.
#include <nvtx3/nvToolsExt.h>

#include <algorithm>

#include "../../include/convnet_b200_conv.h"
#include "../../include/convnet_b200_conv_gemm.h"
#include "../../include/convnet_b200_ext.h"
#include "conv_kernels.h"

using namespace cnb;

namespace {

ConvDesc as_2d(ConvDesc d) { d.kernel_size_t = 1; d.stride_t = 1; d.padding_t = 0; return d; }

// one NVTX range per C-ABI entry (named after the entry point), so an nsys / ncu timeline of a host application shows
// which reference call every kernel belongs to; header-only NVTX3: a no-op costing a few ns when no tool is attached
struct Range {
  explicit Range(const char* name) { nvtxRangePushA(name); }
  ~Range() { nvtxRangePop(); }
};

// ---- dispatch: tensor-core path when the mode and the shape allow, else fp32 CUDA cores
// Writer protocol (stage.cu): drop staged bf16 copies overlapping the target; when the caller asked for a fresh copy
// (convnet_b200_emit_bf16_next) hand the kernel the buffer, and convert in a trailing pass if the kernel did not fill it.
struct Emit {
  float* target; long long n; __nv_bfloat16* buf = nullptr; bool done = false;
  Emit(float* t, long long n_, bool want) : target(t), n(n_) {
    bf16_note_write(t, n_);
    if (want) buf = bf16_emit_slot(t, n_);          // nullptr outside bf16 mode; marked valid: the kernel below fills it
  }
  void attach(Fuse& f) { f.out16 = buf; f.emitted = &done; }
  void finish() { if (buf && !done) bf16_stage(target, n); }     // nobody filled it: one conversion pass (re-validates the slot)
};

// bias gradient requested with the write (convnet_b200_fuse_next_bias_grad): finish from the kernel's per-slice sums, or
// run the column-sum pass when the kernel did not produce them.  rows = images x positions, cols = channels.
void finish_bias_grad(const Fuse& fuse, const float* part, int slices, const float* target, long long rows, int cols) {
  if (!fuse.bias_grad) return;
  if (slices > 0) colsum_finish(part, fuse.bias_grad, cols, slices, fuse.bg_st, fuse.bg_so);
  else cnb_channel_bias_grad(target, fuse.bias_grad, rows, cols, fuse.bg_st, fuse.bg_so);
}

void conv_up(const ConvGeom& g, const float* images, const float* filters, float* targets, float st, float so) {
  Fuse fuse = take_fuse();
  if (!g.conv && fuse.any()) { fprintf(stderr, "convnet_b200: epilogue fusion is not available for untied filters\n"); abort(); }
  CNB_REQUIRE(!fuse.bias_grad, "convUp: a fused bias gradient belongs to a backward call");
  Emit emit(targets, g.out_total, fuse.emit_bf16 != 0);
  emit.attach(fuse);
  bool dropped = false;
  fuse.dropped = &dropped;
  if (!(state().precision != kPrecFP32 && tc_conv_up(g, images, filters, targets, st, so, fuse))) {
    simt_conv_up(g, images, filters, targets, st, so, fuse);
    note_conv(kPathSimt, 0);
  }
  if (fuse.drop_scale != 0.f && !dropped) {        // the kernel could not apply the dropout: one pass, which also (re)writes the bf16 twin
    dropout_apply(targets, g.out_total, fuse.drop_prob, fuse.drop_scale, fuse.drop_seed, emit.buf);
    if (emit.buf) emit.done = true;
  }
  emit.finish();
}

void conv_down(const ConvGeom& g, const float* derivs, const float* filters, float* targets, float st, float so) {
  Fuse fuse = take_fuse();
  if (fuse.prestage) {                             // filters-only preparation of this call (convnet_b200_prestage_next)
    if (state().precision != kPrecFP32) tc_conv_down_prestage(g, derivs, filters);
    return;
  }
  so *= fuse.out_scale;
  // the mask can ride in the epilogue only when one launch produces the final value of every target element
  const bool whole = g.conv && g.frames == 1 && g.cin0 == 0 && g.Cin == g.CinT;
  const float* late_mask = nullptr;
  if (fuse.relu_mask && !whole) { late_mask = fuse.relu_mask; fuse.relu_mask = nullptr; }
  Emit emit(targets, g.img_total, fuse.emit_bf16 != 0);
  if (!late_mask) emit.attach(fuse);               // a late mask changes the values after the kernel: convert afterwards
  if (!(state().precision != kPrecFP32 && tc_conv_down(g, derivs, filters, targets, st, so, fuse))) {
    simt_conv_down(g, derivs, filters, targets, st, so, fuse);
    note_conv(kPathSimt, 0);
  }
  if (late_mask) {
    const long long n4 = g.img_total;             // (cnb_relu_deriv would consume a pending fuse request; none is pending here)
    cnb_relu_deriv(targets, late_mask, n4);
  }
  CNB_REQUIRE(!fuse.bias_grad || g.frames == 1, "convDown: fused bias gradient is 2-D only");
  finish_bias_grad(fuse, nullptr, 0, targets, (long long)g.N * g.W * g.H, g.CinT);
  emit.finish();
}

// reduction split for the CUDA-core wgrad: enough (tile x chunk) blocks to fill the GPU
void simt_outp_auto(const ConvGeom& g, const float* images, const float* derivs, float* targets, float st, float so) {
  const long long tiles = (long long)ceil_div(g.Cout, 128) * ceil_div(g.K, 128);
  const long long want = std::max<long long>(1, (4LL * num_sms()) / tiles);
  long long chunksY = std::min<long long>(g.modY, std::max<long long>(1, want / g.frames));
  // keep the partial-sum scratch below 1 GiB
  const long long elems = (long long)g.Cout * g.K;
  while (chunksY > 1 && elems * chunksY * g.frames * 4 > (1LL << 30)) chunksY--;
  const int rectH = (int)ceil_div<long long>(g.modY, chunksY);
  simt_conv_outp(g, images, derivs, targets, rectH, g.modX, false, st, so);
}

void conv_outp(const ConvGeom& g, const float* images, const float* derivs, float* targets, float st, float so) {
  take_fuse();                                 // a wgrad call has no epilogue to fuse: a pending request must not leak to a later call
  if (!g.conv) {                               // untied: one [Cout x K] block per module
    simt_conv_outp(g, images, derivs, targets, 1, 1, true, st, so);
    note_conv(kPathSimt, 0);
    return;
  }
  if (state().precision != kPrecFP32 && tc_conv_outp(g, images, derivs, targets, st, so)) return;
  simt_outp_auto(g, images, derivs, targets, st, so);
  note_conv(kPathSimt, 0);
}

void do_conv_up(const char* what, cudamat* images, cudamat* filters, cudamat* targets, Shape4D* is, Shape4D* fs,
                Shape4D* ts, ConvDesc d, float st, bool conv) {
  Range nvtx_range(what);
  ConvGeom g = conv_geom(*is, *fs, *ts, images, filters, targets, d, conv, what);
  conv_up(g, images->data_device, filters->data_device, targets->data_device, st, 1.f);
}
void do_conv_down(const char* what, cudamat* derivs, cudamat* filters, cudamat* targets, Shape4D* ds, Shape4D* fs,
                  Shape4D* ts, ConvDesc d, float st, bool conv) {
  Range nvtx_range(what);
  ConvGeom g = conv_geom(*ts, *fs, *ds, targets, filters, derivs, d, conv, what);
  conv_down(g, derivs->data_device, filters->data_device, targets->data_device, st, 1.f);
}
void do_conv_outp(const char* what, cudamat* images, cudamat* derivs, cudamat* targets, Shape4D* is, Shape4D* ds,
                  Shape4D* ts, ConvDesc d, float st, float so, bool conv) {
  Range nvtx_range(what);
  ConvGeom g = conv_geom(*is, *ts, *ds, images, targets, derivs, d, conv, what);
  conv_outp(g, images->data_device, derivs->data_device, targets->data_device, st, so);
}

void do_pool(const char* what, bool is_max, cudamat* images, cudamat* targets, Shape4D* is, Shape4D* ts, ConvDesc d,
             float so) {
  Range nvtx_range(what);
  PoolGeom g = pool_geom(*is, *ts, images, targets, d, what);
  const Fuse fuse = take_fuse();
  Emit emit(targets->data_device, (long long)targets->size[0] * targets->size[1], fuse.emit_bf16 != 0);
  emit.done = pool_forward(g, is_max, images->data_device, targets->data_device, so, emit.buf, fuse.pool_cache != 0);
  emit.finish();
}
void do_max_undo(const char* what, cudamat* images, cudamat* maxGrads, cudamat* maxActs, cudamat* targets,
                 Shape4D* is, Shape4D* gs, ConvDesc d, float st) {
  Range nvtx_range(what);
  PoolGeom g = pool_geom(*is, *gs, images, maxGrads, d, what);
  CNB_REQUIRE(targets->size[0] == g.N && targets->size[1] == images->size[1], what);
  CNB_REQUIRE(maxActs->size[0] == g.N && maxActs->size[1] == maxGrads->size[1], what);
  const Fuse fuse = take_fuse();
  Emit emit(targets->data_device, (long long)targets->size[0] * targets->size[1], fuse.emit_bf16 != 0);
  int slices = 0;
  float* part = fuse.bias_grad ? (float*)workspace(sizeof(float) * (size_t)(g.H + 2) * g.C * g.T) : nullptr;
  emit.done = max_pool_undo(g, images->data_device, maxGrads->data_device, maxActs->data_device, targets->data_device, st,
                            1.f, fuse.relu_mask, emit.buf, g.T == 1 ? part : nullptr, &slices);
  finish_bias_grad(fuse, part, slices, targets->data_device, (long long)g.N * g.W * g.H * g.T, g.C);
  emit.finish();
}
void do_avg_undo(const char* what, cudamat* avgGrads, cudamat* targets, Shape4D* gs, Shape4D* ts, ConvDesc d, float st,
                 float so) {
  Range nvtx_range(what);
  PoolGeom g = pool_geom(*ts, *gs, targets, avgGrads, d, what);
  const Fuse fuse = take_fuse();
  Emit emit(targets->data_device, (long long)targets->size[0] * targets->size[1], fuse.emit_bf16 != 0);
  int slices = 0;
  float* part = fuse.bias_grad ? (float*)workspace(sizeof(float) * (size_t)(g.H + 2) * g.C * g.T) : nullptr;
  emit.done = avg_pool_undo(g, avgGrads->data_device, targets->data_device, st, so, fuse.relu_mask, emit.buf,
                            g.T == 1 ? part : nullptr, &slices);
  finish_bias_grad(fuse, part, slices, targets->data_device, (long long)g.N * g.W * g.H * g.T, g.C);
  emit.finish();
}

ConvDesc sample_desc(Shape4D* is, Shape4D* ts, int factor) {      // gemm.cu:1503-1541
  ConvDesc d;
  d.kernel_size_y = d.kernel_size_x = factor; d.kernel_size_t = 1;
  d.stride_y = d.stride_x = factor; d.stride_t = 1;
  d.padding_y = d.padding_x = d.padding_t = 0;
  d.num_input_channels = is->shape[3]; d.num_output_channels = ts->shape[3];
  d.input_channel_begin = d.output_channel_begin = 0;
  d.input_channel_end = is->shape[3]; d.output_channel_end = ts->shape[3];
  d.num_groups = 1;
  return d;
}

void do_rnorm(const char* what, cudamat* images, cudamat* targets, int F, int sizeF, float a, float b, bool blocked,
              int frames) {
  Range nvtx_range(what);
  CNB_REQUIRE(F > 0 && frames > 0, what);
  const long long els = (long long)images->size[0] * images->size[1];
  CNB_REQUIRE(els % ((long long)F * frames) == 0, what);
  CNB_REQUIRE(targets->size[0] == images->size[0] && targets->size[1] == images->size[1], what);
  const long long L = els / F / frames;          // locations per frame
  // fused epilogue (convnet_b200_fuse_next relu / convnet_b200_emit_bf16_next): in the tile kernel when it applies, else
  // as trailing passes
  const Fuse fuse = take_fuse();
  const bool fusable = rnorm_can_fuse(F);
  Emit emit(targets->data_device, els, fuse.emit_bf16 != 0);
  for (int t = 0; t < frames; t++)               // conv3d_gemm.cu:167-189: independent per frame
    rnorm_forward(images->data_device + (long long)t * L * F, targets->data_device + (long long)t * L * F, L, F, sizeF,
                  a, b, blocked, fusable && fuse.relu, fusable && emit.buf ? emit.buf + (long long)t * L * F : nullptr);
  if (fuse.relu && !fusable) cnb_relu(targets->data_device, els);
  emit.done = fusable;
  emit.finish();
}
void do_rnorm_undo(const char* what, cudamat* outGrads, cudamat* inputs, cudamat* targets, int F, int sizeF, float a,
                   float b, bool blocked, int frames) {
  Range nvtx_range(what);
  CNB_REQUIRE(F > 0 && frames > 0, what);
  const long long els = (long long)inputs->size[0] * inputs->size[1];
  CNB_REQUIRE(els % ((long long)F * frames) == 0, what);
  CNB_REQUIRE(targets->size[0] == inputs->size[0] && targets->size[1] == inputs->size[1], what);
  CNB_REQUIRE(outGrads->size[0] == inputs->size[0] && outGrads->size[1] == inputs->size[1], what);
  const long long L = els / F / frames;
  const Fuse fuse = take_fuse();
  CNB_REQUIRE(!fuse.bias_grad, "ResponseNormCrossMapUndo: no fused bias gradient here");
  Emit emit(targets->data_device, els, fuse.emit_bf16 != 0);
  for (int t = 0; t < frames; t++)
    rnorm_undo(outGrads->data_device + (long long)t * L * F, inputs->data_device + (long long)t * L * F,
               targets->data_device + (long long)t * L * F, L, F, sizeF, a, b, blocked);
  emit.finish();
}

}  // namespace

extern "C" {

// =============================== ABI-1 (cudamat_conv_gemm.cuh) ===============================
void convUpGemm(cudamat* images, cudamat* filters, cudamat* targets, Shape4D* is, Shape4D* fs, Shape4D* ts,
                ConvDesc d, float scaleTargets) {
  do_conv_up("convUpGemm", images, filters, targets, is, fs, ts, as_2d(d), scaleTargets, true);
}
void convDownGemm(cudamat* derivs, cudamat* filters, cudamat* targets, Shape4D* ds, Shape4D* fs, Shape4D* ts,
                  ConvDesc d, float scaleTargets) {
  do_conv_down("convDownGemm", derivs, filters, targets, ds, fs, ts, as_2d(d), scaleTargets, true);
}
void convOutpGemm(cudamat* images, cudamat* derivs, cudamat* targets, Shape4D* is, Shape4D* ds, Shape4D* ts,
                  ConvDesc d, float scaleTargets, float scaleOutput) {
  do_conv_outp("convOutpGemm", images, derivs, targets, is, ds, ts, as_2d(d), scaleTargets, scaleOutput, true);
}
void convInnerpGemm(cudamat*, cudamat*, cudamat*, Shape4D*, Shape4D*, Shape4D*, ConvDesc, float, float) {
  not_implemented("convInnerpGemm", "no caller in the reference's C++ (SURVEY.md 2.3); out of scope");
}
void localUpGemm(cudamat* images, cudamat* filters, cudamat* targets, Shape4D* is, Shape4D* fs, Shape4D* ts,
                 ConvDesc d, float scaleTargets) {
  do_conv_up("localUpGemm", images, filters, targets, is, fs, ts, as_2d(d), scaleTargets, false);
}
void localDownGemm(cudamat* derivs, cudamat* filters, cudamat* targets, Shape4D* ds, Shape4D* fs, Shape4D* ts,
                   ConvDesc d, float scaleTargets) {
  do_conv_down("localDownGemm", derivs, filters, targets, ds, fs, ts, as_2d(d), scaleTargets, false);
}
void localOutpGemm(cudamat* images, cudamat* derivs, cudamat* targets, Shape4D* is, Shape4D* ds, Shape4D* ts,
                   ConvDesc d, float scaleTargets, float scaleOutput) {
  do_conv_outp("localOutpGemm", images, derivs, targets, is, ds, ts, as_2d(d), scaleTargets, scaleOutput, false);
}

void MaxPoolGemm(cudamat* images, cudamat* targets, Shape4D* is, Shape4D* ts, ConvDesc d, float /*scaleTargets*/,
                 float scaleOutput) {
  do_pool("MaxPoolGemm", true, images, targets, is, ts, d, scaleOutput);
}
void AvgPoolGemm(cudamat* images, cudamat* targets, Shape4D* is, Shape4D* ts, ConvDesc d, float /*scaleTargets*/,
                 float scaleOutput) {
  do_pool("AvgPoolGemm", false, images, targets, is, ts, d, scaleOutput);
}
void MaxPoolUndoGemm(cudamat* images, cudamat* maxGrads, cudamat* maxActs, cudamat* targets, Shape4D* is,
                     Shape4D* gs, ConvDesc d, float scaleTargets) {
  do_max_undo("MaxPoolUndoGemm", images, maxGrads, maxActs, targets, is, gs, d, scaleTargets);
}
void MaxPoolRpropGemm(cudamat*, cudamat*, cudamat*, cudamat*, Shape4D*, Shape4D*, ConvDesc, float) {
  not_implemented("MaxPoolRpropGemm", "R-operator has no caller in the reference's C++; out of scope");
}
void AvgPoolUndoGemm(cudamat* avgGrads, cudamat* targets, Shape4D* gs, Shape4D* ts, ConvDesc d, float scaleTargets) {
  do_avg_undo("AvgPoolUndoGemm", avgGrads, targets, gs, ts, d, scaleTargets, 1.f);
}
void UpSampleGemm(cudamat* images, cudamat* targets, Shape4D* is, Shape4D* ts, int factor, float scaleTargets) {
  CNB_REQUIRE(factor >= 1, "UpSampleGemm");
  // up-sampling == avg-pool undo with output scale factor^2 (gemm.cu:1503-1521)
  do_avg_undo("UpSampleGemm", images, targets, is, ts, sample_desc(ts, is, factor), scaleTargets,
              (float)(factor * factor));
}
void DownSampleGemm(cudamat* images, cudamat* targets, Shape4D* is, Shape4D* ts, int factor) {
  CNB_REQUIRE(factor >= 1, "DownSampleGemm");
  do_pool("DownSampleGemm", false, images, targets, is, ts, sample_desc(is, ts, factor), 1.f);
}

void ResponseNormCrossMapGemm(cudamat* images, cudamat* targets, int numFilters, int sizeF, float addScale,
                              float powScale, bool blocked) {
  do_rnorm("ResponseNormCrossMapGemm", images, targets, numFilters, sizeF, addScale, powScale, blocked, 1);
}
void ResponseNormCrossMapUndoGemm(cudamat* outGrads, cudamat* inputs, cudamat* targets, int numFilters, int sizeF,
                                  float addScale, float powScale, bool blocked) {
  do_rnorm_undo("ResponseNormCrossMapUndoGemm", outGrads, inputs, targets, numFilters, sizeF, addScale, powScale,
                blocked, 1);
}
void ResponseNormCrossMapRpropGemm(cudamat*, cudamat*, cudamat*, int, int, float, float, bool) {
  not_implemented("ResponseNormCrossMapRpropGemm", "R-operator has no caller in the reference's C++; out of scope");
}
void Scale(cudamat* mat, float scale) {
  bf16_note_write(mat->data_device, (long long)mat->size[0] * mat->size[1]);
  scale_buffer(mat->data_device, (long long)mat->size[0] * mat->size[1], scale);
}

void convUp3DGemm(cudamat* images, cudamat* filters, cudamat* targets, Shape4D* is, Shape4D* fs, Shape4D* ts,
                  ConvDesc d, float scaleTargets) {
  do_conv_up("convUp3DGemm", images, filters, targets, is, fs, ts, d, scaleTargets, true);
}
void convDown3DGemm(cudamat* derivs, cudamat* filters, cudamat* targets, Shape4D* ds, Shape4D* fs, Shape4D* ts,
                    ConvDesc d, float scaleTargets) {
  do_conv_down("convDown3DGemm", derivs, filters, targets, ds, fs, ts, d, scaleTargets, true);
}
void convOutp3DGemm(cudamat* images, cudamat* derivs, cudamat* targets, Shape4D* is, Shape4D* ds, Shape4D* ts,
                    ConvDesc d, float scaleTargets, float scaleOutput) {
  do_conv_outp("convOutp3DGemm", images, derivs, targets, is, ds, ts, d, scaleTargets, scaleOutput, true);
}
void ResponseNormCrossMap3DGemm(cudamat* images, cudamat* targets, int numFilters, int sizeF, float addScale,
                                float powScale, bool blocked, int image_size_t) {
  do_rnorm("ResponseNormCrossMap3DGemm", images, targets, numFilters, sizeF, addScale, powScale, blocked, image_size_t);
}
void ResponseNormCrossMap3DUndoGemm(cudamat* outGrads, cudamat* inputs, cudamat* targets, int numFilters, int sizeF,
                                    float addScale, float powScale, bool blocked, int image_size_t) {
  do_rnorm_undo("ResponseNormCrossMap3DUndoGemm", outGrads, inputs, targets, numFilters, sizeF, addScale, powScale,
                blocked, image_size_t);
}

// =============================== ABI-2 (cudamat_conv.cuh) ====================================
void SetupTexture(cudamat*) {}   // texture-object cache of cudamat_conv_util.cu: nothing to do on sm_100a

void convUp(cudamat* images, cudamat* filters, cudamat* targets, Shape4D* is, Shape4D* fs, Shape4D* ts, ConvDesc d,
            float scaleTargets) {
  do_conv_up("convUp", images, filters, targets, is, fs, ts, as_2d(d), scaleTargets, true);
}
void localUp(cudamat* images, cudamat* filters, cudamat* targets, Shape4D* is, Shape4D* fs, Shape4D* ts, ConvDesc d,
             float scaleTargets) {
  do_conv_up("localUp", images, filters, targets, is, fs, ts, as_2d(d), scaleTargets, false);
}
void convDown(cudamat* derivs, cudamat* filters, cudamat* targets, Shape4D* ds, Shape4D* fs, Shape4D* ts, ConvDesc d,
              float scaleTargets) {
  do_conv_down("convDown", derivs, filters, targets, ds, fs, ts, as_2d(d), scaleTargets, true);
}
void localDown(cudamat* derivs, cudamat* filters, cudamat* targets, Shape4D* ds, Shape4D* fs, Shape4D* ts, ConvDesc d,
               float scaleTargets) {
  do_conv_down("localDown", derivs, filters, targets, ds, fs, ts, as_2d(d), scaleTargets, false);
}
void convOutp(cudamat* images, cudamat* derivs, cudamat* targets, Shape4D* is, Shape4D* ds, Shape4D* ts, ConvDesc d,
              int partialSumY, int partialSumX, float scaleTargets, float scaleOutput) {
  d = as_2d(d);
  const int modX = ds->shape[1], modY = ds->shape[2];
  if (partialSumY <= 0) partialSumY = modY;
  if (partialSumX <= 0) partialSumX = modX;
  const int chunks = ceil_div(modX, partialSumX) * ceil_div(modY, partialSumY);
  if (chunks == 1) {
    do_conv_outp("convOutp", images, derivs, targets, is, ds, ts, d, scaleTargets, scaleOutput, true);
    return;
  }
  // targets = `chunks` consecutive [Cout x K] blocks: shape {Cout, kx, ky, Cin*chunks} (weightacts.cu:3126-3170)
  CNB_REQUIRE(ts->shape[3] % chunks == 0, "convOutp");
  Shape4D one = *ts; one.shape[3] = ts->shape[3] / chunks;
  ConvGeom g = conv_geom(*is, one, *ds, images, nullptr, derivs, d, true, "convOutp");
  CNB_REQUIRE(targets->size[0] == g.Cout && (long long)targets->size[1] == (long long)g.K * chunks, "convOutp");
  simt_conv_outp(g, images->data_device, derivs->data_device, targets->data_device, partialSumY, partialSumX, true,
                 scaleTargets, scaleOutput);
  note_conv(kPathSimt, 0);
}
void localOutp(cudamat* images, cudamat* derivs, cudamat* targets, Shape4D* is, Shape4D* ds, Shape4D* ts, ConvDesc d,
               float scaleTargets, float scaleOutput) {
  do_conv_outp("localOutp", images, derivs, targets, is, ds, ts, as_2d(d), scaleTargets, scaleOutput, false);
}

void ResponseNormCrossMap(cudamat* images, cudamat* targets, int numFilters, int sizeF, float addScale, float powScale,
                          bool blocked) {
  do_rnorm("ResponseNormCrossMap", images, targets, numFilters, sizeF, addScale, powScale, blocked, 1);
}
void ResponseNormCrossMapUndo(cudamat* outGrads, cudamat* inputs, cudamat* /*acts*/, cudamat* targets, int numFilters,
                              int sizeF, float addScale, float powScale, bool blocked) {
  do_rnorm_undo("ResponseNormCrossMapUndo", outGrads, inputs, targets, numFilters, sizeF, addScale, powScale, blocked, 1);
}
void ResponseNorm(cudamat*, cudamat*, cudamat*, int, int, float, float) {
  not_implemented("ResponseNorm", "within-map response norm: no Edge type reaches it (src/edge.cc:17-60)");
}
void ResponseNormUndo(cudamat*, cudamat*, cudamat*, cudamat*, cudamat*, int, int, float, float) {
  not_implemented("ResponseNormUndo", "within-map response norm: no Edge type reaches it (src/edge.cc:17-60)");
}
void ContrastNorm(cudamat*, cudamat*, cudamat*, cudamat*, int, int, float, float) {
  not_implemented("ContrastNorm", "contrast norm: no Edge type reaches it (src/edge.cc:17-60)");
}
void ContrastNormUndo(cudamat*, cudamat*, cudamat*, cudamat*, cudamat*, int, int, float, float) {
  not_implemented("ContrastNormUndo", "contrast norm: no Edge type reaches it (src/edge.cc:17-60)");
}

void MaxPool(cudamat* images, cudamat* targets, Shape4D* is, Shape4D* ts, ConvDesc d) {
  do_pool("MaxPool", true, images, targets, is, ts, d, 1.f);
}
void AvgPool(cudamat* images, cudamat* targets, Shape4D* is, Shape4D* ts, ConvDesc d) {
  do_pool("AvgPool", false, images, targets, is, ts, d, 1.f);
}
void MaxPoolUndo(cudamat* images, cudamat* maxGrads, cudamat* maxActs, cudamat* targets, Shape4D* is, Shape4D* gs,
                 ConvDesc d, float scaleTargets) {
  do_max_undo("MaxPoolUndo", images, maxGrads, maxActs, targets, is, gs, d, scaleTargets);
}
void AvgPoolUndo(cudamat* avgGrads, cudamat* targets, Shape4D* gs, Shape4D* ts, ConvDesc d, float scaleTargets) {
  do_avg_undo("AvgPoolUndo", avgGrads, targets, gs, ts, d, scaleTargets, 1.f);
}
void UpSample(cudamat* images, cudamat* targets, Shape4D* is, Shape4D* ts, int factor, float scaleTargets) {
  UpSampleGemm(images, targets, is, ts, factor, scaleTargets);
}
void DownSample(cudamat* images, cudamat* targets, Shape4D* is, Shape4D* ts, int factor) {
  DownSampleGemm(images, targets, is, ts, factor);
}
void RGBToYUV(cudamat*, cudamat*) {
  not_implemented("RGBToYUV", "colour-space edge is a 3x3 dot in the reference (rgb_to_yuv_edge.cc); out of scope");
}

}  // extern "C"
