// stage.cu — bf16 operand copies of fp32 tensors (precision mode 2) and their coherence.
//
// In bf16 mode the conv kernels read bf16 copies of their fp32 operands.  A copy is made either by a conversion pass
// (convnet_b200_bf16_stage / _ensure, or inside the conv call when nothing is staged) or — the cheap way — by the kernel
// that PRODUCES the fp32 tensor, which writes the bf16 twin from the same registers (convnet_b200_emit_bf16_next).
//
// Coherence is kept by the library for everything the library writes: every entry point that writes a tensor calls
// bf16_note_write() first, which drops every staged copy that overlaps the written range, and then either emits a fresh
// copy or leaves none.  Only writes the library cannot see (cudaMemcpy, other libraries) need an explicit
// convnet_b200_bf16_invalidate / _stage by the caller.  CONVNET_B200_STAGE_VERIFY=1 re-converts the fp32 source at every
// use of a staged copy and aborts on the first mismatch — the debugging aid for such a missed write.
#include <cuda_bf16.h>

#include <vector>

#include "conv_kernels.h"

namespace cnb {

namespace {

struct Staged {
  const float* src; long long n; __nv_bfloat16* buf; size_t cap; bool valid; unsigned long long tick; int dev;
  int kind;                         // 0: plain bf16 copy; 1: dgrad weight banks (dgrad_weights), `sig` = geometry they were built for;
  unsigned long long sig;           // 2: max-pool tie masks of the pooled tensor `src` (pool_masks_*), `src2` = the pool input
  const float* src2; long long n2;  // kind 2: a write to EITHER tensor makes the masks stale
};
std::vector<Staged>& table() { static std::vector<Staged> t; return t; }
unsigned long long g_tick = 0;
constexpr size_t kMaxStaged = 128;
inline size_t align_up(size_t v) { return (v + 1023) & ~size_t(1023); }
inline bool aligned16(const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; }

__global__ void __launch_bounds__(256) cvt_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, long long n) {
  const long long n8 = n >> 3;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += stride) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(src) + 2 * i), b = __ldg(reinterpret_cast<const float4*>(src) + 2 * i + 1);
    __nv_bfloat162 r0 = __floats2bfloat162_rn(a.x, a.y), r1 = __floats2bfloat162_rn(a.z, a.w);
    __nv_bfloat162 r2 = __floats2bfloat162_rn(b.x, b.y), r3 = __floats2bfloat162_rn(b.z, b.w);
    uint4 o;
    o.x = *reinterpret_cast<uint32_t*>(&r0); o.y = *reinterpret_cast<uint32_t*>(&r1);
    o.z = *reinterpret_cast<uint32_t*>(&r2); o.w = *reinterpret_cast<uint32_t*>(&r3);
    reinterpret_cast<uint4*>(dst)[i] = o;
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 7)) dst[(n8 << 3) + threadIdx.x] = __float2bfloat16_rn(src[(n8 << 3) + threadIdx.x]);
}

// STAGE_VERIFY: count elements whose staged copy differs from a fresh conversion of the fp32 source
__global__ void __launch_bounds__(256) verify_kernel(const float* __restrict__ src, const __nv_bfloat16* __restrict__ copy,
                                                     long long n, unsigned long long* bad) {
  unsigned long long local = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const __nv_bfloat16 want = __float2bfloat16_rn(src[i]);
    const unsigned short a = *reinterpret_cast<const unsigned short*>(&want), b = *reinterpret_cast<const unsigned short*>(copy + i);
    const bool both_nan = (a & 0x7FFF) > 0x7F80 && (b & 0x7FFF) > 0x7F80;
    if (a != b && !both_nan) local++;
  }
  if (local) atomicAdd(bad, local);
}

bool verify_enabled() {
  static const bool on = getenv("CONVNET_B200_STAGE_VERIFY") && getenv("CONVNET_B200_STAGE_VERIFY")[0] == '1';
  return on;
}

void verify(const Staged& e, long long n) {
  static unsigned long long* bad = nullptr;
  if (!bad) CNB_CUDA_CHECK(cudaMallocManaged((void**)&bad, sizeof(*bad)));
  CNB_CUDA_CHECK(cudaStreamSynchronize(state().stream));
  *bad = 0;
  const int grid = (int)std::min<long long>(std::max<long long>(ceil_div<long long>(n, 256), 1), 8LL * num_sms());
  verify_kernel<<<grid, 256, 0, state().stream>>>(e.src, e.buf, n, bad);
  CNB_CUDA_CHECK(cudaStreamSynchronize(state().stream));
  if (*bad != 0) {
    fprintf(stderr, "convnet_b200: STAGE_VERIFY: the staged bf16 copy of tensor %p (%lld floats) is stale in %llu elements: the "
            "tensor was written after it was staged and nobody re-staged or invalidated it\n", (const void*)e.src, n, *bad);
    abort();
  }
}

Staged* find_slot(const float* ptr, int dev, int kind = 0) {
  for (Staged& e : table()) if (e.src == ptr && e.dev == dev && e.kind == kind) return &e;
  return nullptr;
}

// slot for [ptr, ptr+n) with a buffer of at least n bf16; contents undefined, valid == false
Staged* acquire_slot(const float* ptr, long long n, int kind = 0) {
  std::vector<Staged>& t = table();
  const int dev = current_device();
  Staged* slot = find_slot(ptr, dev, kind);
  if (!slot) {
    if (t.size() >= kMaxStaged) {                                       // recycle the least recently used entry
      slot = &t[0];
      for (Staged& e : t) if (e.tick < slot->tick) slot = &e;
    } else {
      t.push_back(Staged{ptr, 0, nullptr, 0, false, 0, dev, kind, 0, nullptr, 0});
      slot = &t.back();
    }
  }
  const size_t bytes = align_up((size_t)n * 2);
  if (slot->cap < bytes || slot->dev != dev) {                          // (a recycled entry may belong to another device)
    if (slot->buf) {
      CNB_CUDA_CHECK(cudaStreamSynchronize(state().stream));
      if (slot->dev != dev) CNB_CUDA_CHECK(cudaSetDevice(slot->dev));
      CNB_CUDA_CHECK(cudaFree(slot->buf));
      if (slot->dev != dev) CNB_CUDA_CHECK(cudaSetDevice(dev));
    }
    slot->buf = nullptr; slot->cap = 0;
    CNB_CUDA_CHECK(cudaMalloc((void**)&slot->buf, bytes));
    slot->cap = bytes;
  }
  slot->src = ptr; slot->n = n; slot->dev = dev; slot->valid = false; slot->tick = ++g_tick; slot->kind = kind; slot->sig = 0;
  slot->src2 = nullptr; slot->n2 = 0;
  return slot;
}


// ---- dgrad weight banks ---------------------------------------------------------------------------------------------
// dgrad is a stride-1 correlation of the output derivative with the flipped filters — one per stride phase (a, b) of the
// input pixel (x = sx*i + a, y = sy*j + b), each phase seeing only the taps congruent to (a + pad) mod stride.  Run in that
// form it uses the fprop kernel (CTA pairs, MN-major B), which needs the filters of a phase as [c fastest][tap''][o]:
//   bank(a,b)[c + Cin*((u' + ku*v') + ku*kv*o)] = w[o, tx = ra + sx*(ku-1-u'), ty = rb + sy*(kv-1-v'), c]
// (reference semantics: cudamat_conv_gemm.cu:684-825, convDown = Sgemm + kContract).  The banks are a permutation of the
// filter tensor (every tap belongs to exactly one phase), built by one small kernel; cached like a bf16 copy when prestaged.
// one 32 x 32 (o, c) tile of one tap per block: coalesced reads along o, coalesced writes along c
__global__ void __launch_bounds__(256) dgrad_bank_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, DgradBanks b,
                                                         int Cin, int Cout, int kx, int ky, int sx, int sy) {
  __shared__ float tile[32][33];
  int z = blockIdx.z, ph = 0;                         // z enumerates (phase, tap'') in bank order
  while (z >= b.phase[ph].ku * b.phase[ph].kv) { z -= b.phase[ph].ku * b.phase[ph].kv; ph++; }
  const DgradPhase& P = b.phase[ph];
  const int T = P.ku * P.kv, u = z % P.ku, v = z / P.ku;
  const int tx = P.rx + sx * (P.ku - 1 - u), ty = P.ry + sy * (P.kv - 1 - v);
  const int o0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int lx = threadIdx.x & 31, ly = threadIdx.x >> 5;         // 32 x 8 threads
  for (int r = ly; r < 32; r += 8) {
    const int c = c0 + r, o = o0 + lx;
    tile[r][lx] = (c < Cin && o < Cout) ? w[o + (long long)Cout * (tx + kx * (ty + ky * c))] : 0.f;
  }
  __syncthreads();
  for (int r = ly; r < 32; r += 8) {
    const int o = o0 + r, c = c0 + lx;
    if (o < Cout && c < Cin) out[P.offset + c + (long long)Cin * (z + (long long)T * o)] = __float2bfloat16_rn(tile[lx][r]);
  }
}

}  // namespace

int dgrad_phases(const ConvGeom& g, DgradBanks* b) {
  const int pad_x = -g.px, pad_y = -g.py;
  b->count = 0;
  long long off = 0;
  for (int pb = 0; pb < g.sy; pb++)
    for (int pa = 0; pa < g.sx; pa++) {
      if (pa >= g.W || pb >= g.H) continue;
      DgradPhase P;
      P.a = pa; P.b = pb;
      P.rx = (pa + pad_x) % g.sx; P.ry = (pb + pad_y) % g.sy;
      P.ku = P.rx < g.kx ? (g.kx - 1 - P.rx) / g.sx + 1 : 0;
      P.kv = P.ry < g.ky ? (g.ky - 1 - P.ry) / g.sy + 1 : 0;
      P.px = (pa + pad_x - P.rx) / g.sx - (P.ku - 1);
      P.py = (pb + pad_y - P.ry) / g.sy - (P.kv - 1);
      P.Wp = (g.W - pa + g.sx - 1) / g.sx; P.Hp = (g.H - pb + g.sy - 1) / g.sy;
      P.offset = off;
      off += (long long)g.Cin * g.Cout * P.ku * P.kv;
      if (b->count >= kMaxDgradPhases) return -1;
      b->phase[b->count++] = P;
    }
  return b->count;
}

// Only banks built on request (convnet_b200_prestage_next: `keep`) stay valid after the call.  Like a staged copy, cached
// banks follow library writes to the filters but not writes the library cannot see, and a caller that overwrites its
// weights by other means (its own optimizer, a cudaMemcpy) never asked to cache anything: banks built inside a convDown
// serve that call alone.  Their buffer stays with the slot, so the next such call rebuilds into it in stream order.
const __nv_bfloat16* dgrad_weights(const float* filters, const ConvGeom& g, const DgradBanks& b, bool keep) {
  const long long n = (long long)g.Cout * g.K;
  unsigned long long sig = 1469598103934665603ULL;
  for (int v : {g.Cin, g.Cout, g.kx, g.ky, g.sx, g.sy, g.px, g.py, g.W, g.H}) sig = (sig ^ (unsigned)v) * 1099511628211ULL;
  const int dev = current_device();
  Staged* e = find_slot(filters, dev, 1);
  if (e && e->valid && e->n == n && e->sig == sig) { e->tick = ++g_tick; return e->buf; }
  e = acquire_slot(filters, n, 1);
  const dim3 grid((unsigned)ceil_div(g.Cout, 32), (unsigned)ceil_div(g.Cin, 32), (unsigned)(g.kx * g.ky));
  dgrad_bank_kernel<<<grid, 256, 0, state().stream>>>(filters, e->buf, b, g.Cin, g.Cout, g.kx, g.ky, g.sx, g.sy);
  count_launch();
  CNB_LAUNCH_CHECK("dgrad_banks");
  e->valid = keep; e->sig = sig;
  return e->buf;
}

namespace {

}  // namespace

bool want_bf16() { return state().precision == kPrecBF16; }

void to_bf16(const float* src, __nv_bfloat16* dst, long long n) {
  static const int dbg = getenv("CONVNET_B200_TC_DEBUG") ? atoi(getenv("CONVNET_B200_TC_DEBUG")) : 0;
  if (dbg & 4) return;
  const long long n8 = n >> 3;
  const int grid = (int)std::min<long long>(std::max<long long>(ceil_div<long long>(n8, 256), 1), 8LL * num_sms());
  cvt_bf16_kernel<<<grid, 256, 0, state().stream>>>(src, dst, n);
  count_launch();
  CNB_LAUNCH_CHECK("cvt_bf16");
}

const __nv_bfloat16* bf16_staged(const float* src, long long n) {          // nullptr: not staged (or too short)
  if (table().empty()) return nullptr;
  const int dev = current_device();
  for (Staged& e : table())
    if (e.valid && e.kind == 0 && e.src == src && e.dev == dev && e.n >= n) {
      e.tick = ++g_tick;
      if (verify_enabled()) verify(e, n);
      return e.buf;
    }
  return nullptr;
}

void bf16_invalidate(const float* ptr) {
  for (Staged& e : table())
    if (ptr == nullptr || e.src == ptr) e.valid = false;
}

void bf16_note_write(const float* ptr, long long n) {
  if (table().empty() || ptr == nullptr) return;
  const int dev = current_device();
  for (Staged& e : table()) {
    if (!e.valid || e.dev != dev) continue;
    if (ptr < e.src + e.n && e.src < ptr + n) e.valid = false;
    else if (e.src2 && ptr < e.src2 + e.n2 && e.src2 < ptr + n) e.valid = false;
  }
}

void bf16_release() {
  if (table().empty()) return;
  CNB_CUDA_CHECK(cudaStreamSynchronize(state().stream));
  const int dev = current_device();
  for (Staged& e : table())
    if (e.buf) {
      if (e.dev != dev) CNB_CUDA_CHECK(cudaSetDevice(e.dev));
      CNB_CUDA_CHECK(cudaFree(e.buf));
      if (e.dev != dev) CNB_CUDA_CHECK(cudaSetDevice(dev));
    }
  table().clear();
}

void bf16_stage(const float* ptr, long long n) {
  if (!want_bf16() || ptr == nullptr || n <= 0 || !aligned16(ptr)) return;
  Staged* slot = acquire_slot(ptr, n);
  to_bf16(ptr, slot->buf, n);
  slot->valid = true;
}

void bf16_ensure(const float* ptr, long long n) {
  if (!want_bf16() || ptr == nullptr || n <= 0) return;
  if (bf16_staged(ptr, n)) return;
  bf16_stage(ptr, n);
}

__nv_bfloat16* bf16_emit_slot(const float* ptr, long long n) {
  if (!want_bf16() || ptr == nullptr || n <= 0 || !aligned16(ptr)) return nullptr;
  Staged* slot = acquire_slot(ptr, n);
  slot->valid = true;            // stream order: the emitting kernel is enqueued before any reader
  return slot->buf;
}

__nv_bfloat16* bf16_refresh_slot(const float* ptr, long long n) {
  if (!want_bf16() || table().empty()) return nullptr;
  Staged* e = find_slot(ptr, current_device(), 0);
  if (!e || e->n != n || !e->buf) return nullptr;
  e->valid = true; e->tick = ++g_tick;
  return e->buf;
}

// max-pool tie masks: one uint16 per pooled element (bit dx + K*dy set where the window element equals the max, bit 15 where
// the max is > 0), written by the forward kernel on request and read by the undo kernel instead of the pool input and output
uint16_t* pool_masks_slot(const float* acts, long long n_out, const float* images, long long n_in, unsigned long long sig) {
  if (acts == nullptr || n_out <= 0) return nullptr;
  Staged* e = acquire_slot(acts, n_out, 2);          // n_out uint16 == n_out bf16-sized elements
  e->src2 = images; e->n2 = n_in; e->sig = sig; e->valid = true;
  return reinterpret_cast<uint16_t*>(e->buf);
}
const uint16_t* pool_masks_find(const float* acts, long long n_out, const float* images, unsigned long long sig) {
  if (table().empty()) return nullptr;
  Staged* e = find_slot(acts, current_device(), 2);
  if (!e || !e->valid || e->n != n_out || e->src2 != images || e->sig != sig) return nullptr;
  e->tick = ++g_tick;
  return reinterpret_cast<const uint16_t*>(e->buf);
}

__nv_bfloat16* begin_write(float* target, long long n, bool want_emit, bool kernel_can_emit) {
  bf16_note_write(target, n);
  if (want_emit && kernel_can_emit) return bf16_emit_slot(target, n);
  return nullptr;
}
void end_write(float* target, long long n, bool want_emit, const __nv_bfloat16* emitted) {
  if (want_emit && !emitted) bf16_stage(target, n);
}

}  // namespace cnb
