// conv_tc.cu — convolution fprop / dgrad / wgrad as implicit GEMMs on the 5th-generation
// tensor cores (tcgen05.mma, accumulators in TMEM) fed by TMA straight from the caller's
// fp32 CHWN buffers.  No im2col buffer, no layout conversion pass, no atomics.
//
// Layout insight (DESIGN.md §3): in the reference layout the IMAGE index n is the
// contiguous axis of every activation tensor (SURVEY.md Appendix A).  A box of 32
// consecutive images x 32 channels at one pixel is therefore a ready-made MN-major
// SWIZZLE_128B UMMA operand atom stack (32 rows of 128 bytes), and zero-fill of
// out-of-range TMA coordinates implements the convolution padding for free.  Filters
// [K x Cout] (Cout contiguous) are MN-major B for fprop and K-major B for dgrad.
//
//   fprop : D[(n,module), o] = sum_{tap,c}  img[n, x(module,tap), y, c] * w[o, tap, c]     A MN-major, B MN-major
//   dgrad : D[(n,pixel), c]  = sum_{tap,o}  der[n, module(pixel,tap), o] * w[o, tap, c]    A MN-major, B K-major
//   wgrad : D[o, c] (per tap)= sum_{module,n} der[n, module, o] * img[n, x, y, c]          A K-major,  B K-major
//
// One persistent CTA per SM, 6 warps: warp 0 = TMA producer, warp 1 = MMA issuer (+TMEM
// allocator), warps 2..5 = epilogue (TMEM -> registers -> coalesced global stores; each thread
// owns one image / one output channel row, so every store instruction writes 128 contiguous bytes).
// Two TMEM accumulator buffers let the epilogue of tile i overlap the main loop of tile i+1.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cudaTypedefs.h>

#include <algorithm>
#include <vector>

#include "conv_kernels.h"
#include "sm100_ptx.cuh"

namespace cnb {

namespace {

constexpr int kThreads = 192;
constexpr int BM = 128;             // GEMM rows per tile  (4 chunks of 32)
constexpr int BK = 32;              // fp32 (tf32) elements of K per pipeline stage (4 UMMA steps of 8); x-mode constant
constexpr int kMaxStages = 8;
constexpr uint32_t kAStageBytes = BM * 128;      // 16 KiB: 128 rows x 128 B (K-major) or chunks x bk rows x 128 B (MN-major)

enum Op { kFprop = 0, kDgrad = 1, kWgrad = 2 };

struct TcParams {
  // operand element type: tf32 = the caller's fp32 buffers as they are; bf16 = bf16 copies made by a conversion pass.
  // A 128-byte smem row holds `chunk` = 32 (tf32) or 64 (bf16) consecutive images / channels; one pipeline stage
  // covers bk = 32 / 64 elements of K (four UMMA steps of 8 / 16) and an m-tile is cpt = 4 / 2 chunks of images.
  int bf16, chunk, chunk_shift, cpt, bk, nbc;   // nbc = ceil(N / chunk)
  int N, nb;                        // images, ceil(N/32)
  int W, H, modX, modY, modules;
  int Cin, Cout;                    // channel sub-range sizes
  int kx, ky, sx, sy, px, py, taps;
  int frames, frame0;               // fprop/wgrad: number of frames; dgrad: the single frame handled by this launch
  int BN, stages, tmem_cols;
  int m_tiles, n_tiles, num_tiles;
  int kc_blocks;                    // ceil(K-side channels / 32)
  // "x mode" for tiny channel counts (Cin < 8, e.g. the RGB first layer): the kx taps of a filter row (padded to 8)
  // take the place of the channel block.  fprop: one K block = (channel c, 4 filter rows) = 4x8 K rows;
  // wgrad: the N tile is (x_ct channels) x (ky rows) x 8 taps, reduced over ALL modules at once.
  int x_mode, x_yblocks, x_ct;
  uint32_t b_tx_bytes;              // bytes the B-operand TMA(s) of one stage actually deliver
  int b_rows;                       // B stage size in 128-byte rows (MN-major B: whole chunks, so >= the columns used)
  // merged requests: when N % 128 == 0 (2-D) the four 32-image chunks of an m-tile are one box over a
  // (32, ..., N/32, ...) view of the tensor; when Cout % 32 == 0 the BN/32 filter chunks are one box likewise.
  int a_merged, b_merged;
  // CTA pairs (tcgen05 cta_group::2): two CTAs of a cluster share one 256 x BN tile; each loads its own 128 rows of A
  // and HALF of B, the leader issues M = 256 MMAs that read both shared memories, each CTA keeps its 128 rows in TMEM.
  int cta2;
  int dbg;                          // CONVNET_B200_TC_DEBUG bits (timing experiments only): 1 = no TMA loads, 2 = no MMAs, 4 = no bf16 conversion
  int m_groups;                     // m-tiles (or o-tiles) per scheduling unit: m_tiles, or ceil(m_tiles/2) with cta2
  int total_chunks;                 // fprop: nbc*modules*frames ; dgrad: nbc*W*H   (< 2^31, checked on the host)
  int splits, units_per_split;      // wgrad: (frame, module-row) units per reduction split;
                                    // fprop/dgrad of 1x1 / FC shapes with few tiles: K blocks per split (split-K)
  long long part_stride;            // fprop/dgrad split-K: floats between the partial outputs of consecutive splits
  float* out;
  __nv_bfloat16* out16;             // optional bf16 twin of `out` (same indexing): convnet_b200_emit_bf16_next
  float st, so;
  const float* bias; int relu;      // fused fprop epilogue: + bias[o], then max(., 0)
  const float* mask;                // fused dgrad epilogue: zero where mask <= 0 (same layout as out)
  // fast fprop epilogue: dropout of the (bias + ReLU'd) result, element index = offset from `out` (Fuse::drop_*); 0 = none
  float drop_prob, drop_scale;
  unsigned long long drop_seed;
  long long out_frame_step;         // fprop: floats between output frames
  uint32_t idesc;
  // fast kernels (tc_fast_kernel): bf16, one-request A tiles, K per pipeline stage = 16 * ksteps elements
  int ksteps;                       // UMMA K-steps per stage: 4 (64 K elements) or 8 (128)
  uint32_t a_stage_bytes;           // 128 rows x (16 * ksteps) bf16
  int b_chunks;                     // fprop: 64-column chunks of B this CTA stages per k-block
  // fast fprop: where output position (i, j) of the modX x modY grid lands in the target tensor: pixel
  // (i*o_sx + o_x0, j*o_sy + o_y0) of an o_W-wide plane of out_plane pixels.  Plain fprop: identity.  dgrad run as a
  // stride-1 correlation per stride phase (tc_conv_down_as_fprop) writes every o_sx-th pixel.
  int o_sx, o_sy, o_x0, o_y0, o_W;
  long long out_plane;
};

struct __align__(8) SmemCtl {
  uint64_t full[kMaxStages];
  uint64_t empty[kMaxStages];
  uint64_t tmem_full[2];
  uint64_t tmem_empty[2];
  uint32_t tmem_base;
  int tile_nkb[16];                 // fast kernels: k-blocks of the tile, producer -> MMA issuer (ring over tiles; the producer runs <= 9 tiles ahead)
};

// ------------------------------------------------------------------------------------------------
// tile / k-block enumeration, shared by the producer (which loads) and the MMA warp (which only counts).
// All 32-bit arithmetic: one thread per CTA walks this, so every division counts.
// ------------------------------------------------------------------------------------------------
struct Tile {
  int m_tile, n_tile;               // fprop/dgrad
  int tap, o_tile, c_tile, split;   // wgrad
};

template <int OP>
__device__ __forceinline__ Tile decode_tile(const TcParams& p, int t, int rank) {
  Tile r;
  if (OP == kWgrad) {
    r.split = t % p.splits; t /= p.splits;
    r.c_tile = t % p.n_tiles; t /= p.n_tiles;
    r.o_tile = t % p.m_groups; t /= p.m_groups;
    if (p.cta2) r.o_tile = 2 * r.o_tile + rank;
    r.tap = t;
    r.m_tile = r.o_tile; r.n_tile = r.c_tile;
  } else {
    r.split = t % p.splits; t /= p.splits;
    r.n_tile = t % p.n_tiles;
    r.m_tile = t / p.n_tiles;
    if (p.cta2) r.m_tile = 2 * r.m_tile + rank;
    r.tap = r.o_tile = r.c_tile = 0;
  }
  return r;
}

// The four 32-row chunks of an fprop/dgrad m-tile: image offset, position (module / pixel) and frame.
struct Chunks {
  int n[4], pos[4], f[4];
  bool ok[4];
};
__device__ __forceinline__ Chunks decode_chunks(const TcParams& p, int m_tile, int per_frame) {
  Chunks c;
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const int q = m_tile * p.cpt + i;
    c.ok[i] = i < p.cpt && q < p.total_chunks;
    const int ib = q % p.nbc, r = q / p.nbc;
    c.n[i] = c.ok[i] ? ib * p.chunk : p.N;   // n >= N: the whole TMA box is out of range -> zero-filled
    c.pos[i] = r % per_frame;
    c.f[i] = c.ok[i] ? r / per_frame : 0;
  }
  return c;
}

// dgrad: module coordinate touched by tap t at input coordinate X, or -1
__device__ __forceinline__ int dgrad_mod(int X, int p, int t, int s, int mods) {
  const int a = X - p - t;
  if (a < 0) return -1;
  const int m = a / s;
  if (m * s != a || m >= mods) return -1;
  return m;
}

// dgrad: per-chunk bit masks of the taps that reach a module along x and along y (kx, ky <= 32)
struct DgradTaps {
  uint32_t xm[4], ym[4];
  __device__ __forceinline__ bool live(int c, int tx, int ty) const { return ((xm[c] >> tx) & (ym[c] >> ty) & 1u) != 0; }
  __device__ __forceinline__ bool any(int tx, int ty) const { return live(0, tx, ty) | live(1, tx, ty) | live(2, tx, ty) | live(3, tx, ty); }
};
__device__ __forceinline__ DgradTaps dgrad_taps(const TcParams& p, const Chunks& ch) {
  DgradTaps d;
#pragma unroll
  for (int c = 0; c < 4; c++) {
    d.xm[c] = d.ym[c] = 0;
    if (!ch.ok[c]) continue;
    const int X = ch.pos[c] % p.W, Y = ch.pos[c] / p.W;
    for (int t = 0; t < p.kx; t++) d.xm[c] |= (dgrad_mod(X, p.px, t, p.sx, p.modX) >= 0 ? 1u : 0u) << t;
    for (int t = 0; t < p.ky; t++) d.ym[c] |= (dgrad_mod(Y, p.py, t, p.sy, p.modY) >= 0 ? 1u : 0u) << t;
  }
  return d;
}
__device__ __forceinline__ int dgrad_live_taps(const TcParams& p, const DgradTaps& d, const DgradTaps& e) {
  int live = 0;
  for (int ty = 0; ty < p.ky; ty++)
    for (int tx = 0; tx < p.kx; tx++) live += (d.any(tx, ty) || e.any(tx, ty)) ? 1 : 0;
  return live;
}

// wgrad: the reduction of one tile runs over rows r = f*modY + my in [r0, r1) and, inside a row, over the
// modules mx in [mx_lo, mx_hi] whose tap lands inside the image (the others contribute zeros and are skipped).
struct WgradSpan { int r0, r1, mx_lo, mx_hi, live_rows; };
__device__ __forceinline__ bool wgrad_row_live(const TcParams& p, int r, int ty) {
  const int Y = (r % p.modY) * p.sy + p.py + ty;
  return (unsigned)Y < (unsigned)p.H;
}
__device__ __forceinline__ WgradSpan wgrad_span(const TcParams& p, const Tile& t) {
  WgradSpan s;
  const int tx = t.tap % p.kx, ty = t.tap / p.kx;
  s.r0 = t.split * p.units_per_split;
  s.r1 = min(s.r0 + p.units_per_split, p.modY * p.frames);
  const int lo = -(p.px + tx);                             // mx*sx >= lo
  s.mx_lo = lo <= 0 ? 0 : (lo + p.sx - 1) / p.sx;
  const int hi = p.W - 1 - p.px - tx;                      // mx*sx <= hi
  s.mx_hi = hi < 0 ? -1 : min(hi / p.sx, p.modX - 1);
  s.live_rows = 0;
  if (s.mx_hi >= s.mx_lo)
    for (int r = s.r0; r < s.r1; r++) s.live_rows += wgrad_row_live(p, r, ty) ? 1 : 0;
  return s;
}

// ------------------------------------------------------------------------------------------------
// PAIR kernels hold only cta_group::2 tcgen05 instructions and MUST be launched as clusters of two (the driver rejects
// a kernel that uses cta_group::2 outside a cluster launch, so the two flavours are separate instantiations).
template <int OP, bool PAIR>
__global__ void __launch_bounds__(kThreads, 1)
tc_conv_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const TcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr bool cta2 = PAIR;
  const int rank = cta2 ? (int)ptx::cluster_ctarank() : 0;          // 0 = leader of the pair
  const int bn_local = cta2 ? p.BN / 2 : p.BN;                      // B columns / rows this CTA stages
  const uint32_t b_stage_bytes = (uint32_t)p.b_rows * 128;
  uint8_t* smemA = smem;
  uint8_t* smemB = smem + (size_t)p.stages * kAStageBytes;
  SmemCtl* ctl = reinterpret_cast<SmemCtl*>(smemB + (size_t)p.stages * b_stage_bytes);

  // warp index through a shuffle: provably warp-uniform, which keeps the role branches and their loops on the uniform path
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; s++) { ptx::mbar_init(&ctl->full[s], 1); ptx::mbar_init(&ctl->empty[s], 1); }
    for (int a = 0; a < 2; a++) { ptx::mbar_init(&ctl->tmem_full[a], 1); ptx::mbar_init(&ctl->tmem_empty[a], cta2 ? 8 : 4); }
    ptx::fence_barrier_init();
    ptx::tma_prefetch_desc(&mapA);
    ptx::tma_prefetch_desc(&mapB);
  }
  if (warp == 1) {
    if constexpr (cta2) { ptx::tmem_alloc_2sm(&ctl->tmem_base, (uint32_t)p.tmem_cols); ptx::tmem_relinquish_2sm(); }
    else { ptx::tmem_alloc(&ctl->tmem_base, (uint32_t)p.tmem_cols); ptx::tmem_relinquish(); }
  }
  ptx::tc_fence_before();
  if constexpr (cta2) ptx::cluster_sync(); else __syncthreads();              // peer barriers are initialised before anyone signals them
  ptx::tc_fence_after();
  ptx::pdl_launch_dependents();       // the kernel queued behind this one may start its prologue (it waits for this grid's end)
  ptx::pdl_wait();                    // ... as this one's just overlapped its predecessor's tail; from here on: global memory
  const int t_first = cta2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int t_step = cta2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const uint32_t tmem_base = ctl->tmem_base;

  if (warp == 0) {
    // =============================== TMA producer ===============================
    {
      const bool elected = ptx::elect_one();             // every lane walks the loops, one lane talks to the TMA unit
      int stage = 0; uint32_t phase = 0;
      const bool no_tma = (p.dbg & 1) != 0;
      const uint32_t tx_bytes = no_tma ? 0u : (kAStageBytes + p.b_tx_bytes) * (cta2 ? 2u : 1u);   // the leader's barrier counts both CTAs
      for (int t = t_first; t < p.num_tiles; t += t_step) {
        const Tile tile = decode_tile<OP>(p, t, rank);
        auto begin_stage = [&]() -> uint8_t* {
          ptx::mbar_wait(&ctl->empty[stage], phase ^ 1);
          if (rank == 0 && elected) ptx::mbar_arrive_expect_tx(&ctl->full[stage], tx_bytes);
          return smemA + (size_t)stage * kAStageBytes;
        };
        // TMA wrappers: in pair mode the completion bytes go to the leader's barrier
        auto lda5 = [&](const void* m, void* dst, int c0, int c1, int c2, int c3, int c4) {
          if (no_tma || !elected) return;
          if constexpr (cta2) ptx::tma_load_5d_2sm(m, &ctl->full[stage], dst, c0, c1, c2, c3, c4);
          else ptx::tma_load_5d(m, &ctl->full[stage], dst, c0, c1, c2, c3, c4);
        };
        auto lda4 = [&](const void* m, void* dst, int c0, int c1, int c2, int c3) {
          if (no_tma || !elected) return;
          if constexpr (cta2) ptx::tma_load_4d_2sm(m, &ctl->full[stage], dst, c0, c1, c2, c3);
          else ptx::tma_load_4d(m, &ctl->full[stage], dst, c0, c1, c2, c3);
        };
        auto lda3 = [&](const void* m, void* dst, int c0, int c1, int c2) {
          if (no_tma || !elected) return;
          if constexpr (cta2) ptx::tma_load_3d_2sm(m, &ctl->full[stage], dst, c0, c1, c2);
          else ptx::tma_load_3d(m, &ctl->full[stage], dst, c0, c1, c2);
        };
        auto end_stage = [&]() { if (++stage == p.stages) { stage = 0; phase ^= 1; } };

        if (OP == kFprop) {
          const Chunks ch = decode_chunks(p, tile.m_tile, p.modules);
          int cX[4], cY[4];
#pragma unroll
          for (int c = 0; c < 4; c++) {
            cX[c] = (ch.pos[c] % p.modX) * p.sx + p.px;
            cY[c] = (ch.pos[c] / p.modX) * p.sy + p.py;
          }
          if (p.x_mode) {
            for (int c = 0; c < p.Cin; c++)
              for (int yb = 0; yb < p.x_yblocks; yb++) {
                uint8_t* a = begin_stage();
                uint8_t* b = smemB + (size_t)stage * b_stage_bytes;
                if (!elected) { end_stage(); continue; }
                if (p.a_merged) {                // dims (n_lo, x, y, n_hi, c): one 16 KiB request
                  ptx::tma_load_5d(&mapA, &ctl->full[stage], a, 0, cX[0], cY[0] + 4 * yb, ch.n[0] >> 5, c);
                } else {
#pragma unroll
                  for (int q = 0; q < 4; q++)    // 8 consecutive x pixels x 4 filter rows of channel c = 32 K rows
                    ptx::tma_load_5d(&mapA, &ctl->full[stage], a + q * (BK * 128), ch.n[q], c, cX[q], cY[q] + 4 * yb, ch.f[q]);
                }
                if (p.b_merged) {                // dims (o_lo, tx, ty, o_hi, c)
                  ptx::tma_load_5d(&mapB, &ctl->full[stage], b, 0, 0, 4 * yb, tile.n_tile * (p.BN >> 5), c);
                } else {
                  for (int j = 0; j < p.BN / 32; j++)   // taps >= kx and rows >= ky are out of range -> zero weights
                    ptx::tma_load_4d(&mapB, &ctl->full[stage], b + j * (BK * 128), tile.n_tile * p.BN + j * 32, 0, 4 * yb, c);
                }
                end_stage();
              }
          } else
          for (int ty = 0; ty < p.ky; ty++)
            for (int tx = 0; tx < p.kx; tx++) {
              const int tap = tx + p.kx * ty;
              // split-K (host: only when taps == 1): this tile reduces K blocks [cb0, cb1)
              const int cb0 = p.splits > 1 ? tile.split * p.units_per_split : 0;
              const int cb1 = p.splits > 1 ? min(cb0 + p.units_per_split, p.kc_blocks) : p.kc_blocks;
              for (int cb = cb0; cb < cb1; cb++) {
                uint8_t* a = begin_stage();
                uint8_t* b = smemB + (size_t)stage * b_stage_bytes;
                if (p.a_merged) {                // dims (n_lo, c, n_hi, x, y): one 16 KiB request
                  lda5(&mapA, a, 0, cb * p.bk, ch.n[0] >> p.chunk_shift, cX[0] + tx, cY[0] + ty);
                } else {
#pragma unroll
                  for (int c = 0; c < 4; c++)
                    if (c < p.cpt) lda5(&mapA, a + c * (p.bk * 128), ch.n[c], cb * p.bk, cX[c] + tx, cY[c] + ty, ch.f[c]);
                }
                const int o0 = tile.n_tile * p.BN + rank * bn_local;      // this CTA's share of the filter columns
                if (p.b_merged) {                // dims (o_lo, c, o_hi, tap)
                  lda4(&mapB, b, 0, cb * p.bk, o0 >> p.chunk_shift, tap);
                } else {
                  for (int j = 0; j < ((bn_local + p.chunk - 1) >> p.chunk_shift); j++)   // a last partial chunk loads whole
                    lda3(&mapB, b + j * (p.bk * 128), o0 + j * p.chunk, tap, cb * p.bk);
                }
                end_stage();
              }
            }
        } else if (OP == kDgrad) {
          const Chunks ch = decode_chunks(p, tile.m_tile, p.W * p.H);
          const DgradTaps taps = dgrad_taps(p, ch);
          // the pair walks the UNION of the two m-tiles' live taps (a tap dead for this CTA loads zeros)
          const DgradTaps peer = cta2 ? dgrad_taps(p, decode_chunks(p, tile.m_tile ^ 1, p.W * p.H)) : taps;
          const bool none = dgrad_live_taps(p, taps, peer) == 0;  // then one all-zero k-block keeps the pipeline uniform
          int cX[4], cY[4];
#pragma unroll
          for (int c = 0; c < 4; c++) { cX[c] = ch.pos[c] % p.W; cY[c] = ch.pos[c] / p.W; }
          for (int ty = 0; ty < p.ky; ty++)
            for (int tx = 0; tx < p.kx; tx++) {
              if (!(taps.any(tx, ty) || peer.any(tx, ty) || (none && tx == 0 && ty == 0))) continue;
              int mx[4], my[4];
#pragma unroll
              for (int c = 0; c < 4; c++) {
                const bool lv = ch.ok[c] && taps.live(c, tx, ty);
                mx[c] = lv ? (cX[c] - p.px - tx) / p.sx : -1;      // -1: out of range -> zeros
                my[c] = lv ? (cY[c] - p.py - ty) / p.sy : -1;
              }
              const int tap = tx + p.kx * ty;
              const int ob0 = p.splits > 1 ? tile.split * p.units_per_split : 0;
              const int ob1 = p.splits > 1 ? min(ob0 + p.units_per_split, p.kc_blocks) : p.kc_blocks;
              for (int ob = ob0; ob < ob1; ob++) {
                uint8_t* a = begin_stage();
                uint8_t* b = smemB + (size_t)stage * b_stage_bytes;
                if (p.a_merged) {                // all four chunks sit on the same pixel: dims (n_lo, o, n_hi, mx, my)
                  lda5(&mapA, a, 0, ob * p.bk, ch.n[0] >> p.chunk_shift, mx[0], my[0]);
                } else {
#pragma unroll
                  for (int c = 0; c < 4; c++)
                    if (c < p.cpt) lda5(&mapA, a + c * (p.bk * 128), ch.n[c], ob * p.bk, mx[c], my[c], p.frame0);
                }
                lda3(&mapB, b, ob * p.bk, tap, tile.n_tile * p.BN + rank * bn_local);
                end_stage();
              }
            }
        } else if (p.x_mode) {
          // reduction over every module of this split's rows; B holds x_ct channels x ky rows x 8 taps
          const int r0 = tile.split * p.units_per_split, r1 = min(r0 + p.units_per_split, p.modY * p.frames);
          const uint32_t c_bytes = (uint32_t)p.ky * 8 * 128;
          for (int r = r0; r < r1; r++) {
            const int f = r / p.modY, my = r % p.modY;
            for (int mx = 0; mx < p.modX; mx++)
              for (int ib = 0; ib < p.nb; ib++) {
                uint8_t* a = begin_stage();
                uint8_t* b = smemB + (size_t)stage * b_stage_bytes;
                if (!elected) { end_stage(); continue; }
                ptx::tma_load_5d(&mapA, &ctl->full[stage], a, ib * 32, mx, my, tile.o_tile * BM, f);
                for (int c = 0; c < p.x_ct; c++)
                  ptx::tma_load_5d(&mapB, &ctl->full[stage], b + c * c_bytes, ib * 32, mx * p.sx + p.px, my * p.sy + p.py,
                                   tile.c_tile * p.x_ct + c, f);
                end_stage();
              }
          }
        } else {
          const WgradSpan sp = wgrad_span(p, tile);
          const int tx = tile.tap % p.kx, ty = tile.tap / p.kx;
          if (sp.live_rows == 0) {                         // nothing to sum: one zero k-block group
            for (int ib = 0; ib < p.nbc; ib++) {
              uint8_t* a = begin_stage();
              uint8_t* b = smemB + (size_t)stage * b_stage_bytes;
              lda5(&mapA, a, ib * p.chunk, 0, 0, tile.o_tile * BM, 0);
              lda5(&mapB, b, ib * p.chunk, -1, -1, tile.c_tile * p.BN + rank * bn_local, 0);
              end_stage();
            }
          } else {
            for (int r = sp.r0; r < sp.r1; r++) {
              if (!wgrad_row_live(p, r, ty)) continue;
              const int f = r / p.modY, my = r % p.modY;
              const int Y = my * p.sy + p.py + ty;
              for (int mx = sp.mx_lo; mx <= sp.mx_hi; mx++) {
                const int X = mx * p.sx + p.px + tx;
                for (int ib = 0; ib < p.nbc; ib++) {
                  uint8_t* a = begin_stage();
                  uint8_t* b = smemB + (size_t)stage * b_stage_bytes;
                  lda5(&mapA, a, ib * p.chunk, mx, my, tile.o_tile * BM, f);
                  lda5(&mapB, b, ib * p.chunk, X, Y, tile.c_tile * p.BN + rank * bn_local, f);
                  end_stage();
                }
              }
            }
          }
        }
      }
    }
  } else if (warp == 1 && rank == 0) {
    // =============================== MMA issuer (leader CTA only in pair mode) ===
    int stage = 0; uint32_t phase = 0;
    int acc = 0; uint32_t acc_phase = 0;
    // operand descriptors.
    //  MN-major tf32 tiles are [chunk][BK rows][128 B] in SWIZZLE_128B_BASE32B: atoms of 4 K-rows x 128 B,
    //    SBO = 512 B between 4-row groups, LBO = chunk stride, one UMMA (K = 8) = two groups = 1 KiB;
    //  K-major tiles are [row][128 B] in SWIZZLE_128B: SBO = 8 rows = 1 KiB, K step = 32 B inside the atom.
    const bool a_mn = (OP != kWgrad), b_mn = (OP == kFprop);
    //  MN-major bf16 tiles are [chunk][bk rows][128 B] in plain SWIZZLE_128B: atoms of 8 K-rows x 128 B (64 elements of
    //    M/N), SBO = 1 KiB between 8-row groups, LBO = chunk stride, one UMMA (K = 16) = two groups = 2 KiB.
    const uint32_t mn_lbo = (uint32_t)p.bk * 128, mn_sbo = p.bf16 ? 1024 : 512, mn_kstep = p.bf16 ? 2048 : 1024;
    const uint32_t mn_lay = p.bf16 ? ptx::kLayoutSw128 : ptx::kLayoutSw128Base32;
    const uint32_t a_lbo = a_mn ? mn_lbo : 16, b_lbo = b_mn ? mn_lbo : 16;
    const uint32_t a_sbo = a_mn ? mn_sbo : 1024, b_sbo = b_mn ? mn_sbo : 1024;
    const uint32_t a_lay = a_mn ? mn_lay : ptx::kLayoutSw128;
    const uint32_t b_lay = b_mn ? mn_lay : ptx::kLayoutSw128;
    const uint32_t a_kstep = a_mn ? mn_kstep : 32, b_kstep = b_mn ? mn_kstep : 32;
    const uint64_t da_base = ptx::make_smem_desc(ptx::smem_u32(smemA), a_lbo, a_sbo, a_lay);
    const uint64_t db_base = ptx::make_smem_desc(ptx::smem_u32(smemB), b_lbo, b_sbo, b_lay);
    const bool elected = ptx::elect_one();               // the warp stays converged; one lane issues
    for (int t = t_first; t < p.num_tiles; t += t_step) {
      const Tile tile = decode_tile<OP>(p, t, rank);
      int nkb;
      if (OP == kFprop) {
        const int kcb = p.splits > 1 ? min(p.units_per_split, p.kc_blocks - tile.split * p.units_per_split) : p.kc_blocks;
        nkb = p.x_mode ? p.Cin * p.x_yblocks : p.taps * kcb;
      } else if (OP == kDgrad) {
        const DgradTaps own = dgrad_taps(p, decode_chunks(p, tile.m_tile, p.W * p.H));
        const DgradTaps peer = cta2 ? dgrad_taps(p, decode_chunks(p, tile.m_tile ^ 1, p.W * p.H)) : own;
        const int kcb = p.splits > 1 ? min(p.units_per_split, p.kc_blocks - tile.split * p.units_per_split) : p.kc_blocks;
        nkb = max(dgrad_live_taps(p, own, peer), 1) * kcb;
      } else if (p.x_mode) {
        const int r0 = tile.split * p.units_per_split, r1 = min(r0 + p.units_per_split, p.modY * p.frames);
        nkb = (r1 - r0) * p.modX * p.nb;
      } else {
        const WgradSpan sp = wgrad_span(p, tile);
        nkb = max(sp.live_rows * (sp.mx_hi - sp.mx_lo + 1), 1) * p.nbc;
      }
      ptx::mbar_wait(&ctl->tmem_empty[acc], acc_phase ^ 1);
      ptx::tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(acc * p.BN);
      for (int kb = 0; kb < nkb; kb++) {
        ptx::mbar_wait(&ctl->full[stage], phase);
        ptx::tc_fence_after();
        if (elected) {
          if (!(p.dbg & 2)) {
            // descriptors differ from the stage-0 / step-0 ones only in the 14-bit start-address field (16-byte units)
            const uint64_t da0 = da_base + (uint32_t)(stage * (int)(kAStageBytes >> 4));
            const uint64_t db0 = db_base + (uint32_t)(stage * (int)(b_stage_bytes >> 4));
#pragma unroll
            for (int ks = 0; ks < 4; ks++) {               // 4 UMMA steps per stage for both element types
              const uint64_t da = da0 + (uint32_t)(ks * (int)(a_kstep >> 4)), db = db0 + (uint32_t)(ks * (int)(b_kstep >> 4));
              const uint32_t accum = (kb | ks) != 0;
              if (p.bf16) {
                if constexpr (cta2) ptx::mma_bf16_2sm(d_tmem, da, db, p.idesc, accum);
                else ptx::mma_bf16(d_tmem, da, db, p.idesc, accum);
              } else {
                if constexpr (cta2) ptx::mma_tf32_2sm(d_tmem, da, db, p.idesc, accum);
                else ptx::mma_tf32(d_tmem, da, db, p.idesc, accum);
              }
            }
          }
          if constexpr (cta2) {                                       // frees the slot / publishes the accumulator in BOTH CTAs
            ptx::mma_commit_2sm(&ctl->empty[stage], 3);
            if (kb == nkb - 1) ptx::mma_commit_2sm(&ctl->tmem_full[acc], 3);
          } else {
            ptx::mma_commit(&ctl->empty[stage]);            // frees the smem slot when these MMAs retire
            if (kb == nkb - 1) ptx::mma_commit(&ctl->tmem_full[acc]);
          }
        }
        __syncwarp();
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  } else if (warp >= 2) {
    // =============================== epilogue ===================================
    const int quarter = warp & 3;                      // TMEM lane quarter this warp may read
    int acc = 0; uint32_t acc_phase = 0;
    for (int t = t_first; t < p.num_tiles; t += t_step) {
      const Tile tile = decode_tile<OP>(p, t, rank);
      // row owned by this thread and the address of its column 0
      float* row_ptr = nullptr;
      long long col_stride = 0;
      int ncols_valid = 0;
      bool direct_scale = true;
      if (OP == kFprop || OP == kDgrad) {
        // this warp's 32 rows are one half (bf16: 64-image chunks) or the whole (tf32) of chunk qc of the tile
        const int q = tile.m_tile * 4 + quarter, sub = p.chunk_shift - 5;
        const int qc = q >> sub, half = q & ((1 << sub) - 1);
        const int per_frame = (OP == kFprop) ? p.modules : p.W * p.H;
        if (qc < p.total_chunks) {
          const int ib = qc % p.nbc, r = qc / p.nbc, pos = r % per_frame, f = r / per_frame;
          const int n = ib * p.chunk + half * 32 + lane;
          if (n < p.N) {
            col_stride = (long long)p.N * per_frame;
            row_ptr = p.out + (OP == kFprop ? f * p.out_frame_step : 0) + n + (long long)p.N * pos +
                      col_stride * ((long long)tile.n_tile * p.BN) + tile.split * p.part_stride;
          }
        }
        ncols_valid = min(p.BN, (OP == kFprop ? p.Cout : p.Cin) - tile.n_tile * p.BN);
        direct_scale = (p.splits == 1);
      } else if (p.x_mode) {
        // column j of the tile = tap tx + 8*(row ty + ky*channel): scattered to dW[o, tx + kx*(ty + ky*c)] below
        const int o = tile.o_tile * BM + quarter * 32 + lane;
        if (o < p.Cout) row_ptr = p.out + (long long)tile.split * p.Cout * p.taps * p.Cin + o;
        ncols_valid = min(p.BN, p.x_ct * p.ky * 8);
        direct_scale = (p.splits == 1);
      } else {
        const int o = tile.o_tile * BM + quarter * 32 + lane;
        const int c0 = tile.c_tile * p.BN;
        col_stride = (long long)p.Cout * p.taps;
        if (o < p.Cout)
          row_ptr = p.out + (long long)tile.split * p.Cout * p.taps * p.Cin + o + (long long)p.Cout * tile.tap + col_stride * c0;
        ncols_valid = min(p.BN, p.Cin - c0);
        direct_scale = (p.splits == 1);
      }
      ptx::mbar_wait(&ctl->tmem_full[acc], acc_phase);
      ptx::tc_fence_after();
      const uint32_t t_addr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * p.BN);
      // three store flavours, chosen once per tile so that the unrolled 32-column bodies stay small (the fully
      // general body thrashed the instruction cache: stall_no_inst dominated the epilogue-bound shapes)
      const float so_eff = direct_scale ? p.so : 1.f;
      const bool rmw = direct_scale && p.st != 0.f;
      const bool scatter = (OP == kWgrad) && p.x_mode;
      const bool fused = (OP == kFprop && (p.bias != nullptr || p.relu)) || (OP == kDgrad && p.mask != nullptr);
      for (int j0 = 0; j0 < ncols_valid; j0 += 32) {
        float v[32];
        ptx::tmem_ld_32x32(t_addr + j0, v);
        ptx::tmem_ld_wait();
        if (row_ptr == nullptr) continue;
        const int nv = ncols_valid - j0;                 // > 0
        if (scatter) {
#pragma unroll
          for (int j = 0; j < 32; j++) {
            const int jg = j0 + j, tx = jg & 7, rr = jg >> 3, ty = rr % p.ky, c = tile.c_tile * p.x_ct + rr / p.ky;
            if (j < nv && tx < p.kx && c < p.Cin) {
              float* dst = row_ptr + (long long)p.Cout * (tx + p.kx * (ty + p.ky * c));
              *dst = rmw ? p.st * (*dst) + so_eff * v[j] : so_eff * v[j];
            }
          }
        } else if (fused) {
          float* dst = row_ptr + col_stride * j0;
          __nv_bfloat16* dst16 = p.out16 ? p.out16 + (dst - p.out) : nullptr;
          // all 32 auxiliary loads (bias values / mask elements) are issued before the first dependent store;
          // interleaving them with the stores serialised one memory latency per column
          float aux[32];
          if (OP == kFprop) {
            const float* bias = p.bias ? p.bias + tile.n_tile * p.BN + j0 : nullptr;
#pragma unroll
            for (int j = 0; j < 32; j++) aux[j] = (bias != nullptr && j < nv) ? __ldg(bias + j) : 0.f;
          } else {
            const float* mp = p.mask + (dst - p.out);
#pragma unroll
            for (int j = 0; j < 32; j++) aux[j] = (j < nv) ? __ldg(mp + col_stride * j) : 1.f;
          }
#pragma unroll
          for (int j = 0; j < 32; j++, dst += col_stride)
            if (j < nv) {
              float r = so_eff * v[j];
              if (rmw) r += p.st * (*dst);
              if (OP == kFprop) {
                r += aux[j];
                if (p.relu) r = fmaxf(r, 0.f);
              } else if (!(aux[j] > 0.f)) r = 0.f;
              *dst = r;
              if (dst16) dst16[col_stride * j] = __float2bfloat16_rn(r);
            }
        } else if (rmw) {
          float* dst = row_ptr + col_stride * j0;
          __nv_bfloat16* dst16 = p.out16 ? p.out16 + (dst - p.out) : nullptr;
#pragma unroll
          for (int j = 0; j < 32; j++, dst += col_stride)
            if (j < nv) {
              const float r = p.st * (*dst) + so_eff * v[j];
              *dst = r;
              if (dst16) dst16[col_stride * j] = __float2bfloat16_rn(r);
            }
        } else {
          float* dst = row_ptr + col_stride * j0;
          __nv_bfloat16* dst16 = p.out16 ? p.out16 + (dst - p.out) : nullptr;
#pragma unroll
          for (int j = 0; j < 32; j++, dst += col_stride)
            if (j < nv) {
              const float r = so_eff * v[j];
              *dst = r;
              if (dst16) dst16[col_stride * j] = __float2bfloat16_rn(r);
            }
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {                                     // the leader's MMA warp owns the accumulator hand-shake
        if (rank == 0) ptx::mbar_arrive(&ctl->tmem_empty[acc]);
        else ptx::mbar_arrive_remote(&ctl->tmem_empty[acc], 0);
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }

  ptx::tc_fence_before();
  if constexpr (cta2) ptx::cluster_sync(); else __syncthreads();              // nobody signals a peer that has already left
  if (warp == 1) {
    ptx::tc_fence_after();
    if constexpr (cta2) ptx::tmem_dealloc_2sm(tmem_base, (uint32_t)p.tmem_cols);
    else ptx::tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}


// ================================================================================================
// tc_fast_kernel — the same three implicit GEMMs, specialised for the shapes the training step spends its time in.
//
// ncu on the general kernel above (profiles/r2_conv2_dgrad_ncu.md) showed where the time goes: NOT the tensor pipe (16-54 %
// active), not L2 (< 30 %), but the single producer warp — 55-80 dependent uniform-datapath instructions per k-block
// (run-time layout switches, 64-bit address arithmetic, per-tap divisions, vote/R2UR traffic around every TMA issue) and the
// same again in the MMA-issuing warp, with the per-tile tap decode on top.  This kernel removes the switches at compile time:
//   * bf16 operands only; every A tile is ONE TMA request (N % 128 == 0); channel counts are multiples of 32;
//     2-D, no split-K, overwrite (scaleTargets == 0); anything else still takes the general kernel;
//   * K per pipeline stage is 64 OR 128 elements (ksteps 4 / 8): half the barrier round trips and TMA issues per flop
//     whenever three 128-deep stages fit in shared memory;
//   * the producer and MMA loops work on 32-bit shared-window addresses that advance by adds; waits have an out-of-line
//     slow path; the producer hands the k-block count of each tile to the MMA warp through shared memory instead of both
//     decoding the tile; dgrad live taps are arithmetic progressions (first tap, count) computed once per tile.
// Pipeline, barriers, TMEM double buffering and the CTA-pair protocol are those of tc_conv_kernel.
// ================================================================================================
struct FastTile {
  int nkb;                          // k-blocks of this tile (>= 1)
  int a2, a3, a4;                   // A coordinates that are fixed for the tile (meaning depends on OP)
  int n0, n1;                       // loop counts of the two outer k-loop levels
  int t0;                           // first tap (dgrad) / unused
  int b0;                           // B coordinate fixed for the tile
};

// XM: the tf32 "x mode" for tiny channel counts (the RGB first layer), see TcParams::x_mode — fprop: one k-block per
// channel = 8 x-taps x 8 filter rows (64 K rows, eight UMMA steps of 8); wgrad: the N tile is (channels x ky rows x 8 taps).
// 10 warps: producer, MMA issuer, and EIGHT epilogue warps — two per TMEM lane quarter, taking alternate 32-column slabs.
// With the main loop no longer the limiter the 1x1 layers became epilogue-bound at ~2.5 TB/s: one warp per scheduler
// cannot keep enough stores / mask loads in flight (profiles/r2_layer_probe_fast_v2_dgrad_as_fprop.log).
constexpr int kFastThreads = 320;
template <int OP, bool PAIR, bool XM>
__global__ void __launch_bounds__(kFastThreads, 1)
tc_fast_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const __grid_constant__ TcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int rank = PAIR ? (int)(blockIdx.x & 1u) : 0;               // clusters are (2,1,1): the rank is the parity of blockIdx.x
  const uint32_t b_stage_bytes = (uint32_t)p.b_rows * 128u;
  uint8_t* smemA = smem;
  uint8_t* smemB = smem + (size_t)p.stages * p.a_stage_bytes;
  SmemCtl* ctl = reinterpret_cast<SmemCtl*>(smemB + (size_t)p.stages * b_stage_bytes);
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; s++) { ptx::mbar_init(&ctl->full[s], 1); ptx::mbar_init(&ctl->empty[s], 1); }
    for (int a = 0; a < 2; a++) { ptx::mbar_init(&ctl->tmem_full[a], 1); ptx::mbar_init(&ctl->tmem_empty[a], PAIR ? 16 : 8); }
    ptx::fence_barrier_init();
    ptx::tma_prefetch_desc(&mapA);
    ptx::tma_prefetch_desc(&mapB);
  }
  if (warp == 1) {
    if constexpr (PAIR) { ptx::tmem_alloc_2sm(&ctl->tmem_base, (uint32_t)p.tmem_cols); ptx::tmem_relinquish_2sm(); }
    else { ptx::tmem_alloc(&ctl->tmem_base, (uint32_t)p.tmem_cols); ptx::tmem_relinquish(); }
  }
  ptx::tc_fence_before();
  if constexpr (PAIR) ptx::cluster_sync(); else __syncthreads();
  ptx::tc_fence_after();
  // everything above touched only shared memory, TMEM and the kernel parameters: with programmatic dependent launch it has
  // overlapped the tail of the previous kernel in the stream; from here on this kernel reads what that kernel wrote
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const int t_first = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int t_step = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const uint32_t tmem_base = ctl->tmem_base;
  const int bn_local = PAIR ? p.BN / 2 : p.BN;
  const int bk = p.ksteps * 16;                                     // K elements per stage
  const uint32_t bar_full0 = ptx::smem_u32(&ctl->full[0]), bar_empty0 = ptx::smem_u32(&ctl->empty[0]);

  if (warp == 0) {
    // =============================== TMA producer ===============================
    const bool elected = ptx::elect_one();
    const uint32_t a_base = ptx::smem_u32(smemA), b_base = ptx::smem_u32(smemB);
    const uint32_t tx_bytes = (p.a_stage_bytes + p.b_tx_bytes) * (PAIR ? 2u : 1u);
    uint32_t stage = 0, phase = 0, a_addr = a_base, b_addr = b_base, bar_off = 0;
    int tcount = 0;
    // one pipeline slot: wait until the MMAs that read it have retired, arm the barrier, return the addresses to fill
#define CNB_STAGE_BEGIN()                                                                              \
    ptx::mbar_wait_a(bar_empty0 + bar_off, phase ^ 1u);                                                \
    const uint32_t fullb = PAIR ? ptx::leader_addr(bar_full0 + bar_off) : (bar_full0 + bar_off);       \
    if (elected && rank == 0) ptx::mbar_arrive_expect_tx_a(bar_full0 + bar_off, tx_bytes);
#define CNB_STAGE_END()                                                                                \
    a_addr += p.a_stage_bytes; b_addr += b_stage_bytes; bar_off += 8;                                  \
    if (++stage == (uint32_t)p.stages) { stage = 0; phase ^= 1u; a_addr = a_base; b_addr = b_base; bar_off = 0; }

    for (int t = t_first; t < p.num_tiles; t += t_step, tcount++) {
      if (OP == kFprop && XM) {
        const int n_tile = t % p.n_tiles, m_tile = t / p.n_tiles;
        const int q = m_tile * 4;                                     // first 32-image chunk of the tile
        const bool ok = q < p.total_chunks;
        const int ib = q % p.nb, pos = q / p.nb;
        const int n_hi = ok ? ib : p.nb;
        const int cX = (pos % p.modX) * p.sx + p.px, cY = (pos / p.modX) * p.sy + p.py;
        if (elected) ctl->tile_nkb[tcount & 15] = p.Cin;
        for (int c = 0; c < p.Cin; c++) {
          CNB_STAGE_BEGIN();
          if (elected) {
            ptx::tma5_a<PAIR>(&mapA, fullb, a_addr, 0, cX, cY, n_hi, c);                          // dims (n_lo, x, y, n_hi, c): 8 x 8 taps
            ptx::tma5_a<PAIR>(&mapB, fullb, b_addr, 0, 0, 0, n_tile * (p.BN >> 5), c);            // dims (o_lo, tx, ty, o_hi, c)
          }
          CNB_STAGE_END();
        }
      } else if (OP == kFprop) {
        const int n_tile = t % p.n_tiles, mg = t / p.n_tiles;
        const int m_tile = PAIR ? 2 * mg + rank : mg;
        const int q = m_tile * 2;                                     // first 64-image chunk of the tile
        const bool ok = q < p.total_chunks;
        const int ib = q % p.nbc, pos = q / p.nbc;
        const int n_hi = ok ? ib : p.nbc;                             // out of range: the whole box zero-fills
        const int cX = (pos % p.modX) * p.sx + p.px, cY = (pos / p.modX) * p.sy + p.py;
        const int o0 = n_tile * p.BN + rank * bn_local;
        if (elected) ctl->tile_nkb[tcount & 15] = p.taps * p.kc_blocks;
        int tap = 0;
        for (int ty = 0; ty < p.ky; ty++)
          for (int tx = 0; tx < p.kx; tx++, tap++)
            for (int c = 0; c < p.Cin; c += bk) {
              CNB_STAGE_BEGIN();
              if (elected) {
                ptx::tma5_a<PAIR>(&mapA, fullb, a_addr, 0, c, n_hi, cX + tx, cY + ty);            // dims (n_lo, c, n_hi, x, y)
                if (p.b_merged) ptx::tma4_a<PAIR>(&mapB, fullb, b_addr, 0, c, o0 >> 6, tap);     // dims (o_lo, c, o_hi, tap)
                else
                  for (int j = 0; j < p.b_chunks; j++)                                             // dims (o, tap, c)
                    ptx::tma3_a<PAIR>(&mapB, fullb, b_addr + (uint32_t)j * (uint32_t)(bk * 128), o0 + j * 64, tap, c);
              }
              CNB_STAGE_END();
            }
      } else if (OP == kDgrad) {
        const int n_tile = t % p.n_tiles, mg = t / p.n_tiles;
        const int m_tile = PAIR ? 2 * mg + rank : mg;
        const int q = m_tile * 2;
        const bool ok = q < p.total_chunks;
        const int ib = q % p.nbc, pos = q / p.nbc;
        const int n_hi = ok ? ib : p.nbc;
        // live taps along x: t = tx0 + i*sx, i < ntx, reading module mx0 - i  (cudamat_conv_gemm.cu:684-825: the gather form
        // of kContract); dead taps are skipped, not multiplied by zero
        const int X = pos % p.W, Y = pos / p.W;
        int tx0, ntx, mx0, ty0, nty, my0;
        {
          const int a = X - p.px;                                      // >= 0 (px <= 0)
          const int lo = max(a - (p.modX - 1) * p.sx, 0);               // smallest tap whose module index is <= modX-1
          const int r = a % p.sx;
          tx0 = lo + ((r - lo) % p.sx + p.sx) % p.sx;                  // first tap >= lo congruent to a (mod sx)
          const int hi = min(p.kx - 1, a);
          ntx = hi >= tx0 ? (hi - tx0) / p.sx + 1 : 0;
          mx0 = (a - tx0) / p.sx;
        }
        {
          const int a = Y - p.py;
          const int lo = max(a - (p.modY - 1) * p.sy, 0);
          const int r = a % p.sy;
          ty0 = lo + ((r - lo) % p.sy + p.sy) % p.sy;
          const int hi = min(p.ky - 1, a);
          nty = hi >= ty0 ? (hi - ty0) / p.sy + 1 : 0;
          my0 = (a - ty0) / p.sy;
        }
        if (!ok || ntx == 0 || nty == 0) { ntx = 1; nty = 1; tx0 = 0; ty0 = 0; mx0 = -1; my0 = -1; }   // one all-zero group
        const int c0 = n_tile * p.BN + rank * bn_local;
        if (elected) ctl->tile_nkb[tcount & 15] = ntx * nty * p.kc_blocks;
        for (int iy = 0; iy < nty; iy++)
          for (int ix = 0; ix < ntx; ix++) {
            const int tap = (tx0 + ix * p.sx) + p.kx * (ty0 + iy * p.sy);
            for (int o = 0; o < p.Cout; o += bk) {
              CNB_STAGE_BEGIN();
              if (elected) {
                ptx::tma5_a<PAIR>(&mapA, fullb, a_addr, 0, o, n_hi, mx0 - ix, my0 - iy);          // dims (n_lo, o, n_hi, mx, my)
                ptx::tma3_a<PAIR>(&mapB, fullb, b_addr, o, tap, c0);                               // dims (o, tap, c): 64 o per panel
                if (p.ksteps == 8) ptx::tma3_a<PAIR>(&mapB, fullb, b_addr + (uint32_t)bn_local * 128u, o + 64, tap, c0);
              }
              CNB_STAGE_END();
            }
          }
      } else if (XM) {
        // x-mode wgrad tile (o_tile, c_tile, split): all modules of the split's rows; B = x_ct channels x ky rows x 8 taps
        int tt = t;
        const int split = tt % p.splits; tt /= p.splits;
        const int c_tile = tt % p.n_tiles; const int o_tile = tt / p.n_tiles;
        const int r0 = split * p.units_per_split, r1 = min(r0 + p.units_per_split, p.modY);
        const int cps = p.ksteps >> 2, nsteps = p.nb / cps;              // 32-image chunks per stage
        if (elected) ctl->tile_nkb[tcount & 15] = max(r1 - r0, 0) * p.modX * nsteps;
        for (int my = r0; my < r1; my++)
          for (int mx = 0; mx < p.modX; mx++)
            for (int ib = 0; ib < nsteps; ib++) {
              CNB_STAGE_BEGIN();
              if (elected) {
                ptx::tma5_a<PAIR>(&mapA, fullb, a_addr, 0, mx, my, o_tile * BM, cps * ib);       // dims (n_lo, mx, my, o, n_hi)
                ptx::tma5_a<PAIR>(&mapB, fullb, b_addr, 0, mx * p.sx + p.px, my * p.sy + p.py, c_tile * p.x_ct, cps * ib);   // (n_lo, x, y, c, n_hi)
              }
              CNB_STAGE_END();
            }
      } else {
        // wgrad tile (tap, o_tile, c_tile, split): sum over the module rows of this split whose tap lands inside the image
        int tt = t;
        const int split = tt % p.splits; tt /= p.splits;
        const int c_tile = tt % p.n_tiles; tt /= p.n_tiles;
        int o_tile = tt % p.m_groups; tt /= p.m_groups;
        if (PAIR) o_tile = 2 * o_tile + rank;
        const int tx = tt % p.kx, ty = tt / p.kx;
        int r0 = split * p.units_per_split, r1 = min(r0 + p.units_per_split, p.modY);
        // rows: 0 <= my*sy + py + ty < H ; columns likewise
        const int ylo = -(p.py + ty), yhi = p.H - 1 - p.py - ty;
        r0 = max(r0, ylo <= 0 ? 0 : (ylo + p.sy - 1) / p.sy);
        r1 = min(r1, yhi < 0 ? 0 : yhi / p.sy + 1);
        const int xlo = -(p.px + tx), xhi = p.W - 1 - p.px - tx;
        const int mx_lo = xlo <= 0 ? 0 : (xlo + p.sx - 1) / p.sx;
        const int mx_hi = xhi < 0 ? -1 : min(xhi / p.sx, p.modX - 1);
        const int nmx = max(mx_hi - mx_lo + 1, 0), nrow = max(r1 - r0, 0);
        const int cps = p.ksteps >> 2;                                  // 64-image chunks per stage (1 or 2)
        const int nsteps = p.nbc / cps;
        const bool none = nmx == 0 || nrow == 0;
        if (elected) ctl->tile_nkb[tcount & 15] = none ? nsteps : nrow * nmx * nsteps;
        const int o0 = o_tile * BM, c0 = c_tile * p.BN + rank * bn_local;
        if (none) {
          for (int ib = 0; ib < nsteps; ib++) {                         // nothing to sum: one group of zero k-blocks
            CNB_STAGE_BEGIN();
            if (elected) {
              ptx::tma5_a<PAIR>(&mapA, fullb, a_addr, 0, -1, -1, o0, cps * ib);
              ptx::tma5_a<PAIR>(&mapB, fullb, b_addr, 0, -1, -1, c0, cps * ib);
            }
            CNB_STAGE_END();
          }
        } else {
          for (int my = r0; my < r1; my++) {
            const int Yc = my * p.sy + p.py + ty;
            for (int mx = mx_lo; mx <= mx_hi; mx++) {
              const int Xc = mx * p.sx + p.px + tx;
              for (int ib = 0; ib < nsteps; ib++) {
                CNB_STAGE_BEGIN();
                if (elected) {
                  ptx::tma5_a<PAIR>(&mapA, fullb, a_addr, 0, mx, my, o0, cps * ib);               // dims (n_lo, mx, my, o, n_hi)
                  ptx::tma5_a<PAIR>(&mapB, fullb, b_addr, 0, Xc, Yc, c0, cps * ib);               // dims (n_lo, x, y, c, n_hi)
                }
                CNB_STAGE_END();
              }
            }
          }
        }
      }
    }
#undef CNB_STAGE_BEGIN
#undef CNB_STAGE_END
  } else if (warp == 1 && rank == 0) {
    // =============================== MMA issuer (leader CTA only in pair mode) ===
    // operand layouts exactly as in tc_conv_kernel; K-steps inside a stage: MN-major operands advance by 16 rows of 128 B,
    // K-major ones by 32 B inside a 64-element panel and by one panel (rows * 128 B) after four steps
    const bool a_mn = (OP != kWgrad), b_mn = (OP == kFprop);
    // MN-major tiles are [chunk][K rows][128 B]: bf16 in SWIZZLE_128B (8-row groups, 16 rows per UMMA step), tf32 (XM) in
    // SWIZZLE_128B_BASE32B (4-row groups, 8 rows per step); LBO = one chunk of K rows
    const uint32_t mn_rows = XM ? 64u : (uint32_t)bk;
    const uint32_t mn_lbo = mn_rows * 128u, mn_sbo = XM ? 512u : 1024u;
    const uint32_t mn_lay = XM ? ptx::kLayoutSw128Base32 : ptx::kLayoutSw128;
    // K-major B rows per panel: the columns of the tile (x-mode wgrad: the x_ct * ky * 8 tap rows the TMA box delivers)
    const uint32_t b_rows_local = (OP == kWgrad && XM) ? (uint32_t)(p.x_ct * p.ky * 8) : (uint32_t)bn_local;
    const uint64_t da_base = ptx::make_smem_desc(ptx::smem_u32(smemA), a_mn ? mn_lbo : 16u, a_mn ? mn_sbo : 1024u, a_mn ? mn_lay : ptx::kLayoutSw128);
    const uint64_t db_base = ptx::make_smem_desc(ptx::smem_u32(smemB), b_mn ? mn_lbo : 16u, b_mn ? mn_sbo : 1024u, b_mn ? mn_lay : ptx::kLayoutSw128);
    // K-step offsets in descriptor units of 16 B: MN-major = the rows of one step (bf16: 16 x 128 B, tf32: 8 x 128 B);
    // K-major = 32 B inside a 128-byte panel row, then one panel (rows x 128 B) after four steps
    const uint32_t mn_step = XM ? 64u : 128u;
    const uint32_t a_lo = a_mn ? mn_step : 2u, a_hi = a_mn ? 4u * mn_step : (uint32_t)(BM * 128 >> 4);
    const uint32_t b_lo = b_mn ? mn_step : 2u, b_hi = b_mn ? 4u * mn_step : (b_rows_local * 128u) >> 4;
    const uint32_t a_stage_u = p.a_stage_bytes >> 4, b_stage_u = b_stage_bytes >> 4;
    const bool elected = ptx::elect_one();
    uint32_t stage = 0, phase = 0, bar_off = 0, a_off = 0, b_off = 0;
    uint32_t acc = 0, acc_phase = 0;
    int tcount = 0;
    const uint32_t tfull0 = ptx::smem_u32(&ctl->tmem_full[0]), tempty0 = ptx::smem_u32(&ctl->tmem_empty[0]);
    for (int t = t_first; t < p.num_tiles; t += t_step, tcount++) {
      ptx::mbar_wait_a(tempty0 + acc * 8, acc_phase ^ 1u);
      ptx::tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * (uint32_t)p.BN;
      int nkb = 1;
      for (int kb = 0; kb < nkb; kb++) {
        ptx::mbar_wait_a(bar_full0 + bar_off, phase);
        if (kb == 0) nkb = *reinterpret_cast<volatile int*>(&ctl->tile_nkb[tcount & 15]);     // published before the tile's first TMA
        ptx::tc_fence_after();
        if (elected) {
          const uint64_t da0 = da_base + a_off, db0 = db_base + b_off;
#pragma unroll
          for (int ks = 0; ks < 4; ks++) {
            if constexpr (XM) ptx::mma_tf32_a<PAIR>(d_tmem, da0 + ks * a_lo, db0 + ks * b_lo, p.idesc, (uint32_t)((kb | ks) != 0));
            else ptx::mma_bf16_a<PAIR>(d_tmem, da0 + ks * a_lo, db0 + ks * b_lo, p.idesc, (uint32_t)((kb | ks) != 0));
          }
          if (p.ksteps == 8) {
#pragma unroll
            for (int ks = 0; ks < 4; ks++) {
              if constexpr (XM) ptx::mma_tf32_a<PAIR>(d_tmem, da0 + a_hi + ks * a_lo, db0 + b_hi + ks * b_lo, p.idesc, 1u);
              else ptx::mma_bf16_a<PAIR>(d_tmem, da0 + a_hi + ks * a_lo, db0 + b_hi + ks * b_lo, p.idesc, 1u);
            }
          }
          ptx::mma_commit_a<PAIR>(bar_empty0 + bar_off);                                  // frees the slot (both CTAs in pair mode)
          if (kb == nkb - 1) ptx::mma_commit_a<PAIR>(tfull0 + acc * 8);
        }
        __syncwarp();
        a_off += a_stage_u; b_off += b_stage_u; bar_off += 8;
        if (++stage == (uint32_t)p.stages) { stage = 0; phase ^= 1u; a_off = 0; b_off = 0; bar_off = 0; }
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
  } else if (warp >= 2) {
    // =============================== epilogue ===================================
    const int quarter = warp & 3;                      // TMEM lane quarter this warp may read (warp id mod 4)
    const int slab0 = ((warp - 2) >> 2) * 32;            // warps 2-5 take slabs 0, 2, 4, ...; warps 6-9 slabs 1, 3, 5, ...
    uint32_t acc = 0, acc_phase = 0;
    const uint32_t tfull0 = ptx::smem_u32(&ctl->tmem_full[0]), tempty0 = ptx::smem_u32(&ctl->tmem_empty[0]);
    for (int t = t_first; t < p.num_tiles; t += t_step) {
      float* row_ptr = nullptr;
      long long col_stride;
      int ncols, col0;
      if (OP == kFprop || OP == kDgrad) {
        const int n_tile = t % p.n_tiles, mg = t / p.n_tiles;
        const int m_tile = PAIR ? 2 * mg + rank : mg;
        // this warp's 32 rows: half of one 64-image chunk (bf16), or one whole 32-image chunk (tf32 x mode)
        const int qc = XM ? m_tile * 4 + quarter : m_tile * 2 + (quarter >> 1);
        col_stride = (OP == kFprop) ? (long long)p.N * p.out_plane : (long long)p.N * p.W * p.H;
        col0 = n_tile * p.BN;
        ncols = min(p.BN, (OP == kFprop ? p.Cout : p.Cin) - col0);
        if (qc < p.total_chunks) {
          const int cpp = XM ? p.nb : p.nbc;                          // chunks per position
          const int ib = qc % cpp, pos = qc / cpp;
          const int n = XM ? ib * 32 + lane : ib * 64 + (quarter & 1) * 32 + lane;
          long long opos = pos;
          if (OP == kFprop) {
            const int i = pos % p.modX, j = pos / p.modX;
            opos = (long long)(j * p.o_sy + p.o_y0) * p.o_W + i * p.o_sx + p.o_x0;
          }
          row_ptr = p.out + n + (long long)p.N * opos + col_stride * col0;
        }
      } else {
        int tt = t;
        const int split = tt % p.splits; tt /= p.splits;
        const int c_tile = tt % p.n_tiles; tt /= p.n_tiles;
        int o_tile = XM ? tt : tt % p.m_groups;                      // x mode has no tap level: tt is the o tile
        if (!XM) tt /= p.m_groups;
        if (PAIR) o_tile = 2 * o_tile + rank;
        const int o = o_tile * BM + quarter * 32 + lane;
        col0 = c_tile * p.BN;
        col_stride = (long long)p.Cout * p.taps;
        ncols = min(p.BN, p.Cin - col0);
        if (XM) {                                                    // tile = (o_tile, c_tile, split); columns are (tap, row, channel)
          col0 = c_tile * p.x_ct;
          ncols = p.x_ct * p.ky * 8;
          if (o < p.Cout) row_ptr = p.out + (long long)split * p.Cout * p.taps * p.Cin + o;
        } else if (o < p.Cout)
          row_ptr = p.out + (long long)split * p.Cout * p.taps * p.Cin + o + (long long)p.Cout * tt + col_stride * col0;
      }
      ptx::mbar_wait_a(tfull0 + acc * 8, acc_phase);
      ptx::tc_fence_after();
      const uint32_t t_addr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * (uint32_t)p.BN;
      for (int j0 = slab0; j0 < ncols; j0 += 64) {                   // ncols is a multiple of 32 (host)
        float v[32];
        ptx::tmem_ld_32x32(t_addr + j0, v);
        ptx::tmem_ld_wait();
        if (row_ptr == nullptr) continue;
        float* dst = row_ptr + col_stride * j0;
        __nv_bfloat16* dst16 = p.out16 ? p.out16 + (dst - p.out) : nullptr;
        if (OP == kFprop) {
          float bv[32];
          const float* bp = p.bias ? p.bias + col0 + j0 : nullptr;
#pragma unroll
          for (int j = 0; j < 32; j++) bv[j] = bp ? __ldg(bp + j) : 0.f;
          const bool relu = p.relu != 0;
          if (p.mask == nullptr) {
            const bool drop = p.drop_scale != 0.f;
            unsigned long long ctr = p.drop_seed + (unsigned long long)(dst - p.out);      // seed + element index
#pragma unroll
            for (int j = 0; j < 32; j++) {
              float r = fmaf(p.so, v[j], bv[j]);
              r = relu ? fmaxf(r, 0.f) : r;
              if (drop) { r *= dropout_keep(ctr, p.drop_prob, p.drop_scale); ctr += (unsigned long long)col_stride; }
              *dst = r;
              if (dst16) { *dst16 = __float2bfloat16_rn(r); dst16 += col_stride; }
              dst += col_stride;
            }
          } else {                                                   // dgrad in fprop form: ReLU' of the layer receiving the derivative
            float mk[32];
            const float* mp = p.mask + (dst - p.out);
#pragma unroll
            for (int j = 0; j < 32; j++) { mk[j] = __ldg(mp); mp += col_stride; }
#pragma unroll
            for (int j = 0; j < 32; j++) {
              float r = fmaf(p.so, v[j], bv[j]);
              r = mk[j] > 0.f ? r : 0.f;
              *dst = r;
              if (dst16) { *dst16 = __float2bfloat16_rn(r); dst16 += col_stride; }
              dst += col_stride;
            }
          }
        } else if (OP == kDgrad) {
          float mk[32];
          const float* mp = p.mask ? p.mask + (dst - p.out) : nullptr;
#pragma unroll
          for (int j = 0; j < 32; j++) { mk[j] = mp ? __ldg(mp) : 1.f; if (mp) mp += col_stride; }
#pragma unroll
          for (int j = 0; j < 32; j++) {
            const float r = mk[j] > 0.f ? p.so * v[j] : 0.f;
            *dst = r;
            if (dst16) { *dst16 = __float2bfloat16_rn(r); dst16 += col_stride; }
            dst += col_stride;
          }
        } else if (XM) {
          // column jg = tap tx + 8 * (row ty + ky * channel): scattered to dW[o, tx + kx*(ty + ky*c)]
#pragma unroll
          for (int j = 0; j < 32; j++) {
            const int jg = j0 + j, tx = jg & 7, rr = jg >> 3, ty = rr % p.ky, c = col0 + rr / p.ky;
            if (jg < ncols && tx < p.kx && c < p.Cin) row_ptr[(long long)p.Cout * (tx + p.kx * (ty + p.ky * c))] = p.so * v[j];
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; j++) { *dst = p.so * v[j]; dst += col_stride; }
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (rank == 0) ptx::mbar_arrive_a(tempty0 + acc * 8);
        else ptx::mbar_arrive_remote_a(tempty0 + acc * 8, 0);
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
  }

  ptx::tc_fence_before();
  if constexpr (PAIR) ptx::cluster_sync(); else __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    if constexpr (PAIR) ptx::tmem_dealloc_2sm(tmem_base, (uint32_t)p.tmem_cols);
    else ptx::tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
PFN_cuTensorMapEncodeTiled_v12000 encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    CNB_CUDA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres));
    CNB_REQUIRE(qres == cudaDriverEntryPointSuccess && ptr != nullptr, "cuTensorMapEncodeTiled");
    fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(ptr);
  }
  return fn;
}

// operand element type of one launch (see TcParams)
struct Elem { int bf16, esz, chunk, shift, bk; };
inline Elem elem_for(bool bf16) { return bf16 ? Elem{1, 2, 64, 6, 64} : Elem{0, 4, 32, 5, 32}; }

// tensor map over fp32 or bf16 data; dims[0] is the contiguous axis; strides in ELEMENTS for dims 1..rank-1
bool make_map(CUtensorMap* map, const void* base, const Elem& e, int rank, const long long* dims, const long long* strides,
              const int* box, bool mn_major) {
  cuuint64_t gdim[5], gstr[4];
  cuuint32_t bdim[5], estr[5];
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) return false;
  for (int i = 0; i < rank; i++) {
    if (dims[i] <= 0 || dims[i] > 0xFFFFFFFFLL) return false;
    gdim[i] = (cuuint64_t)dims[i];
    bdim[i] = (cuuint32_t)box[i];
    estr[i] = 1;
    if (box[i] > 256) return false;
    if (i > 0) {
      const long long bytes = strides[i - 1] * e.esz;
      if (bytes % 16 != 0 || bytes <= 0 || bytes >= (1LL << 40)) return false;
      gstr[i - 1] = (cuuint64_t)bytes;
    }
  }
  // 32-bit MN-major operands need the 32-byte-atom flavour of the 128-byte swizzle (UMMA SWIZZLE_128B_BASE32B)
  const CUtensorMapSwizzle sw = (mn_major && !e.bf16) ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B;
  CUresult r = encode_fn()(map, e.bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank,
                           const_cast<void*>(base), gdim, gstr, bdim, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    fprintf(stderr, "convnet_b200: cuTensorMapEncodeTiled failed (%d)\n", (int)r);
    return false;
  }
  return true;
}

int pick_bn(int cols, int granule) {              // N-tile: as wide as possible, <= 256, balanced across tiles
  const int tiles = ceil_div(cols, 256);
  const int bn = ceil_div(ceil_div(cols, tiles), granule) * granule;
  return std::min(256, std::max(granule, bn));
}

int tmem_cols_for(int bn) { int c = 32; while (c < 2 * bn) c *= 2; return c; }

size_t smem_bytes_for(int bn, int stages) {
  return 1024 + (size_t)stages * (kAStageBytes + (size_t)bn * 128) + sizeof(SmemCtl) + 16;
}

int pick_stages(int bn) {
  int s = kMaxStages;
  while (s > 2 && smem_bytes_for(bn, s) > 225 * 1024) s--;
  return s;
}

template <int OP>
void launch(const CUtensorMap& a, const CUtensorMap& b, TcParams& p) {
  if (p.b_rows == 0) p.b_rows = p.cta2 ? p.BN / 2 : p.BN;
  p.stages = pick_stages(p.b_rows);
  p.tmem_cols = tmem_cols_for(p.BN);
  const size_t smem = smem_bytes_for(p.b_rows, p.stages);
  // the attribute belongs to the (function, device) pair: set it once per device this process launches on
  static unsigned long long attr_devices = 0;
  const int dev = current_device();
  if (dev >= 64 || !((attr_devices >> dev) & 1ULL)) {
    CNB_CUDA_CHECK(cudaFuncSetAttribute(tc_conv_kernel<OP, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CNB_CUDA_CHECK(cudaFuncSetAttribute(tc_conv_kernel<OP, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    if (dev < 64) attr_devices |= 1ULL << dev;
  }
  if (p.cta2) {
    // one cluster of two CTAs (one TPC) per scheduling unit; persistent over the pair tiles
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2u * (unsigned)std::min(p.num_tiles, num_sms() / 2));
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = state().stream;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = pdl_enabled() ? 2 : 1;
    CNB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, tc_conv_kernel<OP, true>, a, b, p));
  } else {
    const int grid = std::min(p.num_tiles, num_sms());
    launch_pdl(tc_conv_kernel<OP, false>, dim3((unsigned)grid), dim3(kThreads), smem, state().stream, a, b, p);
  }
  count_launch();
  CNB_LAUNCH_CHECK("tc_conv");
}

// CTA-pair mode (see TcParams::cta2). Worth it when the grid is full anyway: the pair halves the B bytes each SM
// stages per k-block, and these kernels are bound by shared-memory fill rate, not by the tensor pipe.
// `half_granule`: what BN/2 must be a multiple of (32-column atoms for MN-major B, 8 rows for K-major B).
bool pair_enabled() {
  static int en = -1;
  if (en < 0) { const char* e = getenv("CONVNET_B200_NO_2CTA"); en = (e && e[0] == '1') ? 0 : 1; }
  return en == 1;
}
void apply_pair(TcParams& p, int op, int half_granule, long long outer) {
  p.cta2 = 0; p.m_groups = p.m_tiles;
  // measured (profiles/): fprop gains 2-6 %, wgrad up to 48 % (conv2) when the o-tiles pair up evenly, dgrad loses
  static const int ops = getenv("CONVNET_B200_2CTA_OPS") ? atoi(getenv("CONVNET_B200_2CTA_OPS")) : 5;
  if (!pair_enabled() || !((ops >> op) & 1) || p.x_mode || p.m_tiles < 2) return;
  if (op == kWgrad && (p.m_tiles & 1)) return;                     // an odd o-tile count would idle one CTA of the last pair
  if (p.BN % (2 * half_granule) != 0 || p.BN < 2 * half_granule) return;
  const long long pair_tiles = outer * ceil_div(p.m_tiles, 2) * p.n_tiles * p.splits;
  if (pair_tiles < num_sms() / 2) return;                          // small problems keep every SM on its own tile
  p.cta2 = 1;
  p.m_groups = ceil_div(p.m_tiles, 2);
  p.num_tiles = (int)pair_tiles;
  p.b_tx_bytes = (uint32_t)(p.BN / 2) * 128;
  p.idesc = (p.idesc & ~(0x1Fu << 24)) | ((uint32_t)(2 * BM >> 4) << 24);   // M = 256
}


// ---- fast kernels: eligibility, stage shape, launch ------------------------------------------------------------
bool fast_enabled() {
  static const bool off = getenv("CONVNET_B200_NO_FAST") && getenv("CONVNET_B200_NO_FAST")[0] == '1';
  return !off;
}
size_t fast_smem_bytes(size_t a_stage, size_t b_stage, int stages) {
  return 1024 + (size_t)stages * (a_stage + b_stage) + sizeof(SmemCtl) + 16;
}
// K per stage: 128 elements (ksteps 8) when at least three such stages fit, else 64; b_rows_per_kstep4 = 128-byte rows of B
// per 64 K elements.  Returns false if not even two 64-deep stages fit.
bool fast_pick_stages(TcParams& p, int b_rows_per_kstep4) {
  static const int force = getenv("CONVNET_B200_FAST_KSTEPS") ? atoi(getenv("CONVNET_B200_FAST_KSTEPS")) : 0;
  for (int ksteps : {8, 4}) {
    if (force && ksteps != force) continue;
    const size_t a = (size_t)4096 * ksteps, b = (size_t)b_rows_per_kstep4 * (ksteps / 4) * 128;
    int stages = kMaxStages;
    while (stages > 1 && fast_smem_bytes(a, b, stages) > 225 * 1024) stages--;
    if (stages >= (ksteps == 8 && !force ? 3 : 2)) {
      p.ksteps = ksteps; p.a_stage_bytes = (uint32_t)a; p.b_rows = (int)(b / 128); p.b_tx_bytes = (uint32_t)b; p.stages = stages;
      return true;
    }
  }
  return false;
}
template <int OP, bool XM = false>
void launch_fast(const CUtensorMap& a, const CUtensorMap& b, TcParams& p) {
  p.tmem_cols = tmem_cols_for(p.BN);
  const size_t smem = fast_smem_bytes(p.a_stage_bytes, (size_t)p.b_rows * 128, p.stages);
  static unsigned long long attr_devices = 0;
  const int dev = current_device();
  if (dev >= 64 || !((attr_devices >> dev) & 1ULL)) {
    CNB_CUDA_CHECK(cudaFuncSetAttribute(tc_fast_kernel<OP, false, XM>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    if (!XM)
      CNB_CUDA_CHECK(cudaFuncSetAttribute(tc_fast_kernel<OP, !XM, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    if (dev < 64) attr_devices |= 1ULL << dev;
  }
  // programmatic dependent launch: the kernel's prologue (barrier init, TMEM allocation, descriptor prefetch) may run while
  // the previous kernel of the stream drains; it waits (griddepcontrol.wait) before its first global access
  const bool pdl = pdl_enabled();
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(kFastThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = state().stream;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (pdl) { attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization; attr[na].val.programmaticStreamSerializationAllowed = 1; na++; }
  if (p.cta2) {
    if constexpr (!XM) {
      cfg.gridDim = dim3(2u * (unsigned)std::min(p.num_tiles, num_sms() / 2));
      attr[na].id = cudaLaunchAttributeClusterDimension;
      attr[na].val.clusterDim.x = 2; attr[na].val.clusterDim.y = 1; attr[na].val.clusterDim.z = 1;
      na++;
      cfg.attrs = attr; cfg.numAttrs = na;
      CNB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, tc_fast_kernel<OP, !XM, false>, a, b, p));
    }
  } else {
    cfg.gridDim = dim3((unsigned)std::min(p.num_tiles, num_sms()));
    cfg.attrs = attr; cfg.numAttrs = na;
    CNB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, tc_fast_kernel<OP, false, XM>, a, b, p));
  }
  count_launch();
  CNB_LAUNCH_CHECK("tc_fast");
}

bool tc_enabled() {
  static int en = -1;
  if (en < 0) { const char* e = getenv("CONVNET_B200_DISABLE_TC"); en = (e && e[0] == '1') ? 0 : 1; }
  return en == 1 && state().precision >= kPrecTF32;
}
bool allow_merge() {
  static const bool v = !(getenv("CONVNET_B200_NO_TMA_MERGE") && getenv("CONVNET_B200_NO_TMA_MERGE")[0] == '1');
  return v;
}

void fill_common(TcParams& p, const ConvGeom& g, const Elem& e) {
  p.bf16 = e.bf16; p.chunk = e.chunk; p.chunk_shift = e.shift; p.cpt = BM / e.chunk; p.bk = e.bk;
  p.N = g.N; p.nb = ceil_div(g.N, 32); p.nbc = ceil_div(g.N, e.chunk);
  p.W = g.W; p.H = g.H; p.modX = g.modX; p.modY = g.modY; p.modules = g.modules;
  p.Cin = g.Cin; p.Cout = g.Cout;
  p.kx = g.kx; p.ky = g.ky; p.sx = g.sx; p.sy = g.sy; p.px = g.px; p.py = g.py; p.taps = g.kx * g.ky;
  p.frames = g.frames; p.frame0 = 0;
  p.splits = 1; p.units_per_split = 0; p.part_stride = 0;
  p.x_mode = 0; p.x_yblocks = 0; p.x_ct = 0; p.b_tx_bytes = 0; p.b_rows = 0;
  p.a_merged = 0; p.b_merged = 0;
  p.cta2 = 0; p.m_groups = 0;
  static const int dbg = getenv("CONVNET_B200_TC_DEBUG") ? atoi(getenv("CONVNET_B200_TC_DEBUG")) : 0;
  p.dbg = dbg;
  p.bias = nullptr; p.relu = 0; p.mask = nullptr; p.out16 = nullptr;
  p.drop_prob = 0.f; p.drop_scale = 0.f; p.drop_seed = 0;
  p.o_sx = p.o_sy = 1; p.o_x0 = p.o_y0 = 0; p.o_W = g.modX; p.out_plane = g.modules;
  p.ksteps = 4; p.a_stage_bytes = kAStageBytes; p.b_chunks = 0;
  p.out_frame_step = g.out_frame_step;
  p.total_chunks = 0;
}

// image-like tensor (N, W, H, C[, frames]) as a 5-D map ordered (n, c, x, y, f) or (n, x, y, c, f)
bool image_map(CUtensorMap* m, const void* base, const Elem& e, const ConvGeom& g, int Wd, int Hd, int C,
               long long frame_step, bool channel_second, int box_c) {
  const long long N = g.N;
  if (channel_second) {
    const long long dims[5] = {N, C, Wd, Hd, g.frames};
    const long long str[4] = {N * Wd * Hd, N, N * Wd, frame_step};
    const int box[5] = {e.chunk, box_c, 1, 1, 1};
    return make_map(m, base, e, 5, dims, str, box, true);
  }
  const long long dims[5] = {N, Wd, Hd, C, g.frames};
  const long long str[4] = {N, N * Wd, N * Wd * Hd, frame_step};
  const int box[5] = {e.chunk, 1, 1, box_c, 1};
  return make_map(m, base, e, 5, dims, str, box, false);
}

// (n_lo = chunk, channel / x / y ..., n_hi = N/chunk) view for one-request A tiles; `x_mode`: box {32, 8x, 4y, 4 n_hi, 1c}
bool merged_image_map(CUtensorMap* m, const void* base, const Elem& e, const ConvGeom& g, int Wd, int Hd, int C, bool x_mode) {
  const long long N = g.N;
  if (x_mode) {
    const long long dims[5] = {32, Wd, Hd, N / 32, C};
    const long long str[4] = {N, N * Wd, 32, N * Wd * Hd};
    const int box[5] = {32, 8, 4, 4, 1};
    return make_map(m, base, e, 5, dims, str, box, true);
  }
  const long long dims[5] = {e.chunk, C, N / e.chunk, Wd, Hd};
  const long long str[4] = {N * Wd * Hd, e.chunk, N, N * Wd};
  const int box[5] = {e.chunk, e.bk, BM / e.chunk, 1, 1};
  return make_map(m, base, e, 5, dims, str, box, true);
}

inline size_t align_up(size_t v) { return (v + 1023) & ~size_t(1023); }

// ---- split-K for 1x1 / FC shapes: too few output tiles to fill the GPU, long K ------------------------
// out = st*out + so * sum_s part[s]  (+ bias[channel], ReLU | zero where mask <= 0): the fused epilogue moves here
__global__ void __launch_bounds__(256) reduce_split_kernel(const float4* __restrict__ part, float4* out, long long elems4,
                                                           long long stride4, int splits, float st, float so,
                                                           const float* __restrict__ bias, long long per_channel4, int relu,
                                                           const float4* __restrict__ mask) {
  pdl_wait();
  pdl_trigger();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < elems4; i += (long long)gridDim.x * blockDim.x) {
    float4 s = part[i];
    for (int k = 1; k < splits; k++) {
      const float4 v = part[i + k * stride4];
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    s.x *= so; s.y *= so; s.z *= so; s.w *= so;
    if (st != 0.f) { const float4 o = out[i]; s.x += st * o.x; s.y += st * o.y; s.z += st * o.z; s.w += st * o.w; }
    if (bias) { const float b = __ldg(bias + i / per_channel4); s.x += b; s.y += b; s.z += b; s.w += b; }
    if (relu) { s.x = fmaxf(s.x, 0.f); s.y = fmaxf(s.y, 0.f); s.z = fmaxf(s.z, 0.f); s.w = fmaxf(s.w, 0.f); }
    if (mask) {
      const float4 m = mask[i];
      if (!(m.x > 0.f)) s.x = 0.f;
      if (!(m.y > 0.f)) s.y = 0.f;
      if (!(m.z > 0.f)) s.z = 0.f;
      if (!(m.w > 0.f)) s.w = 0.f;
    }
    out[i] = s;
  }
}
void reduce_split(const float* part, float* out, long long elems, int splits, float st, float so, const float* bias,
                  long long per_channel, int relu, const float* mask) {
  const long long e4 = elems / 4;
  const int grid = (int)std::min<long long>(std::max<long long>(ceil_div<long long>(e4, 256), 1), 8LL * num_sms());
  launch_pdl(reduce_split_kernel, dim3((unsigned)grid), dim3(256), 0, state().stream, (const float4*)part, (float4*)out, e4, e4, splits,
             st, so, bias, per_channel / 4, relu, (const float4*)mask);
  count_launch();
  CNB_LAUNCH_CHECK("reduce_split");
}
// how many K splits a fprop/dgrad launch should use (1 = none): only 1x1 / FC shapes that leave most SMs idle
int pick_ksplit(const TcParams& p, const ConvGeom& g, long long out_elems) {
  static const bool off = getenv("CONVNET_B200_NO_SPLITK") && getenv("CONVNET_B200_NO_SPLITK")[0] == '1';
  if (off || p.x_mode || p.taps != 1 || g.frames != 1 || out_elems % 4 != 0) return 1;
  if (p.num_tiles * 2 > num_sms() || p.kc_blocks < 8) return 1;
  const int want = std::min(num_sms() / p.num_tiles, p.kc_blocks / 4);
  return std::max(want, 1);
}
inline bool aligned16(const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; }

}  // namespace

// ---- fprop ---------------------------------------------------------------------------------------
// `bf` selects bf16 operands (CONVNET_B200_PRECISION=bf16): images and filters are first rounded to bf16 copies in
// library scratch, then the same kernel runs kind::f16 MMAs at twice the tf32 rate on half the operand bytes.
static bool tc_conv_up_impl(const ConvGeom& g, const float* images, const float* filters, float* targets, float st, float so,
                            const Fuse& fuse, bool bf) {
  const Elem e = elem_for(bf);
  if (g.N % 4 != 0 || g.Cout % 4 != 0) return false;                        // TMA stride alignment
  const bool x_mode = g.Cin < 8;                                            // tiny channel counts: taps take the K block
  if (x_mode && (g.kx > 8 || g.ky > 8)) return false;
  if (bf && (x_mode || g.N % 8 != 0 || g.Cout % 8 != 0 || !aligned16(images) || !aligned16(filters))) return false;
  // few GEMM rows (FC layers at training batch sizes): the call streams the weights once and is HBM-bound on them; a bf16
  // conversion pass inside the call would read them a second time, so such shapes take bf16 only when the caller keeps a
  // staged bf16 copy of the weights (the training host does: cnb_sgd_momentum refreshes it in the same pass that updates
  // them) — then the call streams HALF the bytes
  if (bf && (long long)g.N * g.modules * g.frames < 1024 && !bf16_staged(filters, (long long)g.Cout * g.K)) return false;
  TcParams p; fill_common(p, g, e);
  p.BN = pick_bn(g.Cout, e.chunk);
  static const int bn_override = getenv("CONVNET_B200_FPROP_BN") ? atoi(getenv("CONVNET_B200_FPROP_BN")) : 0;   // experiments
  if (bn_override >= e.chunk && bn_override <= 256 && bn_override % e.chunk == 0 && !x_mode) p.BN = bn_override;
  p.kc_blocks = ceil_div(g.Cin, e.bk);
  p.x_mode = x_mode ? 1 : 0;
  p.x_yblocks = ceil_div(g.ky, 4);
  p.b_tx_bytes = (uint32_t)p.BN * 128;
  const long long chunks = (long long)p.nb * g.modules * g.frames;
  if (chunks * 4 >= (1LL << 31)) return false;
  p.total_chunks = p.nbc * g.modules * g.frames;
  p.m_tiles = ceil_div(p.total_chunks, p.cpt);
  p.n_tiles = ceil_div(g.Cout, p.BN);
  p.num_tiles = p.m_tiles * p.n_tiles;
  float* const out = targets + (long long)g.cout0 * g.modules * g.N;
  const float* const bias = fuse.bias ? fuse.bias + g.cout0 : nullptr;
  const long long out_elems = (long long)g.Cout * g.modules * g.N;
  const int ks = pick_ksplit(p, g, out_elems);
  if (ks > 1) {
    p.units_per_split = ceil_div(p.kc_blocks, ks);
    p.splits = ceil_div(p.kc_blocks, p.units_per_split);
    p.part_stride = out_elems;
    p.num_tiles *= p.splits;
  }
  const size_t part_bytes = p.splits > 1 ? align_up(sizeof(float) * out_elems * p.splits) : 0;
  p.out = out;
  p.st = st; p.so = so;
  p.bias = bias; p.relu = fuse.relu;
  p.idesc = ptx::make_idesc(bf ? 1 : 2, true, true, BM, p.BN);
  apply_pair(p, kFprop, 32, 1);
  const int bn_local = p.cta2 ? p.BN / 2 : p.BN;
  // MN-major B is staged in whole chunks; a half tile that ends inside a chunk (bf16: BN = 192 -> 96 = 1.5 chunks) loads
  // the rest of that chunk too (never read by the MMA) and cannot use the merged (o_lo, .., o_hi) view
  p.b_rows = ceil_div(bn_local, e.chunk) * e.chunk;
  if (p.cta2) p.b_tx_bytes = (uint32_t)p.b_rows * 128;
  CUtensorMap ma, mb;
  const long long img_off = (long long)g.cin0 * g.H * g.W * g.N;
  const void* img = images + img_off;
  const void* flt = filters;
  const long long taps = (long long)g.kx * g.ky;
  uint8_t* ws = nullptr;
  if (bf) {
    const __nv_bfloat16* si = bf16_staged(images, g.img_total);
    const __nv_bfloat16* sf = bf16_staged(filters, (long long)g.Cout * g.K);
    const size_t ib = si ? 0 : align_up((size_t)g.img_total * 2), fb = sf ? 0 : align_up((size_t)g.Cout * g.K * 2);
    if (part_bytes + ib + fb) ws = (uint8_t*)workspace(part_bytes + ib + fb);
    if (!si) { to_bf16(images, (__nv_bfloat16*)(ws + part_bytes), g.img_total); si = (const __nv_bfloat16*)(ws + part_bytes); }
    if (!sf) { to_bf16(filters, (__nv_bfloat16*)(ws + part_bytes + ib), (long long)g.Cout * g.K); sf = (const __nv_bfloat16*)(ws + part_bytes + ib); }
    img = si + img_off;
    flt = sf;
  } else if (part_bytes) {
    ws = (uint8_t*)workspace(part_bytes);
  }
  if (p.splits > 1) { p.out = (float*)ws; p.bias = nullptr; p.relu = 0; }   // partial sums; the epilogue moves to reduce_split
  // bf16 twin of the output from the same registers: only when this launch writes the final value of EVERY element
  const bool emit = fuse.out16 != nullptr && p.splits == 1 && g.cout0 == 0 && g.Cout == g.CoutT;
  if (emit) p.out16 = fuse.out16;
  p.a_merged = (allow_merge() && g.frames == 1 && g.N % 128 == 0) ? 1 : 0;
  p.b_merged = (allow_merge() && g.Cout % e.chunk == 0 && bn_local % e.chunk == 0) ? 1 : 0;
  // frames of a 3-D conv start in_frame_step floats apart and see Cin (= Cin3d*kt) channels
  if (x_mode) {
    const long long N = g.N;
    if (p.a_merged) {
      if (!merged_image_map(&ma, img, e, g, g.W, g.H, g.Cin, true)) return false;
    } else {
      const long long adims[5] = {N, g.Cin, g.W, g.H, g.frames};
      const long long astr[4] = {N * g.W * g.H, N, N * g.W, g.in_frame_step};
      const int abox[5] = {32, 1, 8, 4, 1};                     // 8 x-taps x 4 filter rows of one channel
      if (!make_map(&ma, img, e, 5, adims, astr, abox, true)) return false;
    }
    if (p.b_merged) {
      const long long bdims[5] = {32, g.kx, g.ky, g.Cout / 32, g.Cin};
      const long long bstr[4] = {g.Cout, (long long)g.Cout * g.kx, 32, (long long)g.Cout * taps};
      const int bbox[5] = {32, 8, 4, p.BN / 32, 1};
      if (!make_map(&mb, flt, e, 5, bdims, bstr, bbox, true)) return false;
    } else {
      const long long bdims[4] = {g.Cout, g.kx, g.ky, g.Cin};
      const long long bstr[3] = {g.Cout, (long long)g.Cout * g.kx, (long long)g.Cout * taps};
      const int bbox[4] = {32, 8, 4, 1};
      if (!make_map(&mb, flt, e, 4, bdims, bstr, bbox, true)) return false;
    }
  } else {
    if (p.a_merged) {
      if (!merged_image_map(&ma, img, e, g, g.W, g.H, g.Cin, false)) return false;
    } else if (!image_map(&ma, img, e, g, g.W, g.H, g.Cin, g.in_frame_step, true, e.bk)) return false;
    if (p.b_merged) {
      const long long dims[4] = {e.chunk, g.Cin, g.Cout / e.chunk, taps};
      const long long str[3] = {(long long)g.Cout * taps, e.chunk, g.Cout};
      const int box[4] = {e.chunk, e.bk, bn_local / e.chunk, 1};
      if (!make_map(&mb, flt, e, 4, dims, str, box, true)) return false;
    } else {
      const long long dims[3] = {g.Cout, taps, g.Cin};
      const long long str[2] = {g.Cout, (long long)g.Cout * taps};
      const int box[3] = {e.chunk, 1, e.bk};
      if (!make_map(&mb, flt, e, 3, dims, str, box, true)) return false;
    }
  }
  bool done = false;
  int kern = 0;
  // the lean kernel takes the shapes the training step lives in (see tc_fast_kernel); the rest stays on the general one
  if (bf && fast_enabled() && !x_mode && p.a_merged && p.splits == 1 && st == 0.f && g.Cout % 32 == 0 && p.BN % 32 == 0) {
    TcParams f = p;
    f.b_chunks = ceil_div(bn_local, 64);
    f.b_merged = (g.Cout % 64 == 0 && bn_local % 64 == 0 && p.BN % 64 == 0) ? 1 : 0;
    if (fast_pick_stages(f, f.b_chunks * 64)) {
      Elem e2 = e; e2.bk = f.ksteps * 16;
      f.kc_blocks = ceil_div(g.Cin, e2.bk);
      CUtensorMap fa, fb;
      bool ok = merged_image_map(&fa, img, e2, g, g.W, g.H, g.Cin, false);
      if (ok && f.b_merged) {
        const long long dims[4] = {64, g.Cin, g.Cout / 64, taps};
        const long long str[3] = {(long long)g.Cout * taps, 64, g.Cout};
        const int box[4] = {64, e2.bk, f.b_chunks, 1};
        ok = make_map(&fb, flt, e2, 4, dims, str, box, true);
      } else if (ok) {
        const long long dims[3] = {g.Cout, taps, g.Cin};
        const long long str[2] = {g.Cout, (long long)g.Cout * taps};
        const int box[3] = {64, 1, e2.bk};
        ok = make_map(&fb, flt, e2, 3, dims, str, box, true);
      }
      if (ok) {
        // dropout in the epilogue: the element index is the offset from the start of the WHOLE target tensor
        const bool drop = fuse.drop_scale != 0.f && g.cout0 == 0 && g.Cout == g.CoutT;
        if (drop) { f.drop_prob = fuse.drop_prob; f.drop_scale = fuse.drop_scale; f.drop_seed = fuse.drop_seed; }
        launch_fast<kFprop>(fa, fb, f);
        done = true;
        kern = kKernLean | kKernAMerged | (f.cta2 ? kKernPair : 0) | (f.b_merged ? kKernBMerged : 0);
        if (drop && fuse.dropped) *fuse.dropped = true;
      }
    }
  }
  // tf32 x mode (RGB first layer) on the lean kernel: one k-block per channel = 8 x 8 taps
  if (!done && !bf && x_mode && fast_enabled() && p.a_merged && p.splits == 1 && st == 0.f && !p.cta2 && g.Cout % 32 == 0 &&
      p.BN % 32 == 0) {
    TcParams f = p;
    f.ksteps = 8; f.a_stage_bytes = 32768; f.b_rows = 2 * p.BN; f.b_tx_bytes = (uint32_t)f.b_rows * 128;
    int stages = kMaxStages;
    while (stages > 1 && fast_smem_bytes(f.a_stage_bytes, (size_t)f.b_rows * 128, stages) > 225 * 1024) stages--;
    f.stages = stages;
    const long long N = g.N;
    const long long adims[5] = {32, g.W, g.H, N / 32, g.Cin}, astr[4] = {N, N * g.W, 32, N * g.W * g.H};
    const int abox[5] = {32, 8, 8, 4, 1};
    const long long bdims[5] = {32, g.kx, g.ky, g.Cout / 32, g.Cin}, bstr[4] = {g.Cout, (long long)g.Cout * g.kx, 32, (long long)g.Cout * taps};
    const int bbox[5] = {32, 8, 8, p.BN / 32, 1};
    CUtensorMap fa, fb;
    if (stages >= 2 && make_map(&fa, img, e, 5, adims, astr, abox, true) && make_map(&fb, flt, e, 5, bdims, bstr, bbox, true)) {
      launch_fast<kFprop, true>(fa, fb, f);
      done = true;
      kern = kKernLean | kKernXMode | kKernAMerged | kKernBMerged;   // both operands through the o-chunked 5-D views
    }
  }
  if (!done) {
    launch<kFprop>(ma, mb, p);
    kern = (p.cta2 ? kKernPair : 0) | (x_mode ? kKernXMode : 0) | (p.splits > 1 ? kKernSplit : 0) |
           (p.a_merged ? kKernAMerged : 0) | (p.b_merged ? kKernBMerged : 0);
  }
  if (emit && fuse.emitted) *fuse.emitted = true;
  if (p.splits > 1) reduce_split((const float*)ws, out, out_elems, p.splits, st, so, bias, (long long)g.modules * g.N, fuse.relu, nullptr);
  note_conv(bf ? kPathTcBf16 : kPathTcTf32, kern);
  return true;
}
bool tc_conv_up(const ConvGeom& g, const float* images, const float* filters, float* targets, float st, float so,
                const Fuse& fuse) {
  if (!tc_enabled() || !g.conv) return false;
  if (want_bf16() && tc_conv_up_impl(g, images, filters, targets, st, so, fuse, true)) return true;
  return tc_conv_up_impl(g, images, filters, targets, st, so, fuse, false);
}


// ---- dgrad in fprop form ---------------------------------------------------------------------------------------------
// dInput[n, x, y, c] = sum_{o, taps} der[n, module, o] * w[o, tap, c] is, for the input pixels of one stride phase, a STRIDE-1
// correlation of the derivative with the phase's flipped taps (stage.cu: dgrad_weights).  In that form it is exactly the fprop
// GEMM — A = derivative (MN-major, one request per tile), B = filter bank [c][tap''][o] (MN-major) — and runs on the fprop
// flavour of tc_fast_kernel: CTA pairs, both operands MN-major, no dead taps.  The gather kernel above, with its K-major B
// of 256 rows per k-block per CTA, measured L2-feed-bound at 0.2-0.4 of the fprop rate on the same problem
// (profiles/r2_layer_probe_fast_v1.log).  One launch per stride phase; the epilogue writes every sx-th / sy-th pixel.
// does the phase-decomposed dgrad (below) take this call?  `banks` receives the phases
static bool dgrad_as_fprop_eligible(const ConvGeom& g, const float* derivs, const float* filters, DgradBanks* banks) {
  static const bool off = getenv("CONVNET_B200_NO_DGRAD_AS_FPROP") && getenv("CONVNET_B200_NO_DGRAD_AS_FPROP")[0] == '1';
  if (off || !fast_enabled() || !g.conv || g.frames != 1) return false;
  if (g.cin0 != 0 || g.Cin != g.CinT || g.cout0 != 0 || g.Cout != g.CoutT) return false;
  if (g.N % 128 != 0 || g.Cin % 32 != 0 || g.Cout % 8 != 0 || !aligned16(derivs) || !aligned16(filters)) return false;
  if ((long long)g.N * g.W * g.H < 1024) return false;                      // FC-shaped: weight-streaming bound, stays tf32
  if (dgrad_phases(g, banks) <= 0) return false;
  for (int i = 0; i < banks->count; i++) if (banks->phase[i].ku == 0 || banks->phase[i].kv == 0) return false;
  return true;
}

void tc_conv_down_prestage(const ConvGeom& g, const float* derivs, const float* filters) {
  DgradBanks banks;
  if (!tc_enabled() || !g.conv || !want_bf16() || !dgrad_as_fprop_eligible(g, derivs, filters, &banks)) return;
  dgrad_weights(filters, g, banks, true);
}

static bool tc_conv_down_as_fprop(const ConvGeom& g, const float* derivs, const float* filters, float* targets, float so,
                                  const Fuse& fuse) {
  DgradBanks banks;
  if (!dgrad_as_fprop_eligible(g, derivs, filters, &banks)) return false;
  const Elem e = elem_for(true);
  // the derivative as bf16 (staged by the producer, or converted here)
  const __nv_bfloat16* sd = bf16_staged(derivs, g.out_total);
  if (!sd) {
    __nv_bfloat16* tmp = (__nv_bfloat16*)workspace(align_up((size_t)g.out_total * 2));
    to_bf16(derivs, tmp, g.out_total);
    sd = tmp;
  }
  const __nv_bfloat16* bank = dgrad_weights(filters, g, banks, false);
  bool emitted_all = fuse.out16 != nullptr;
  int kern = kKernDgradAsFprop | kKernLean | kKernAMerged | (banks.count << kKernPhaseShift);
  for (int i = 0; i < banks.count; i++) {
    const DgradPhase& P = banks.phase[i];
    TcParams p; fill_common(p, g, e);
    // the GEMM of this phase: rows = (image, phase pixel), K = (tap'', o), columns = input channels
    p.modX = P.Wp; p.modY = P.Hp; p.modules = P.Wp * P.Hp;
    p.W = g.modX; p.H = g.modY;                        // the tensor A is read from (the derivative grid)
    p.kx = P.ku; p.ky = P.kv; p.taps = P.ku * P.kv; p.sx = p.sy = 1; p.px = P.px; p.py = P.py;
    p.Cin = g.Cout; p.Cout = g.Cin;
    p.BN = pick_bn(g.Cin, 32);
    p.total_chunks = p.nbc * p.modules;
    p.m_tiles = ceil_div(p.total_chunks, p.cpt);
    p.n_tiles = ceil_div(g.Cin, p.BN);
    p.num_tiles = p.m_tiles * p.n_tiles;
    p.out = targets; p.st = 0.f; p.so = so;
    p.mask = fuse.relu_mask; p.out16 = fuse.out16;
    p.o_sx = g.sx; p.o_sy = g.sy; p.o_x0 = P.a; p.o_y0 = P.b; p.o_W = g.W; p.out_plane = (long long)g.W * g.H;
    p.idesc = ptx::make_idesc(1, true, true, BM, p.BN);
    apply_pair(p, kFprop, 16, 1);
    const int bn_local = p.cta2 ? p.BN / 2 : p.BN;
    p.b_chunks = ceil_div(bn_local, 64);
    p.b_merged = (g.Cin % 64 == 0 && bn_local % 64 == 0 && p.BN % 64 == 0) ? 1 : 0;
    if (!fast_pick_stages(p, p.b_chunks * 64)) return false;
    Elem e2 = e; e2.bk = p.ksteps * 16;
    p.kc_blocks = ceil_div(g.Cout, e2.bk);
    ConvGeom gd = g;                                   // merged_image_map only reads N from the geometry
    CUtensorMap fa, fb;
    if (!merged_image_map(&fa, sd, e2, gd, g.modX, g.modY, g.Cout, false)) return false;
    const __nv_bfloat16* wb = bank + P.offset;
    bool ok;
    if (p.b_merged) {
      const long long dims[4] = {64, g.Cout, g.Cin / 64, p.taps};
      const long long str[3] = {(long long)g.Cin * p.taps, 64, g.Cin};
      const int box[4] = {64, e2.bk, p.b_chunks, 1};
      ok = make_map(&fb, wb, e2, 4, dims, str, box, true);
    } else {
      const long long dims[3] = {g.Cin, p.taps, g.Cout};
      const long long str[2] = {g.Cin, (long long)g.Cin * p.taps};
      const int box[3] = {64, 1, e2.bk};
      ok = make_map(&fb, wb, e2, 3, dims, str, box, true);
    }
    if (!ok) { CNB_REQUIRE(i == 0, "dgrad-as-fprop: tensor map failed after the first phase"); return false; }
    launch_fast<kFprop>(fa, fb, p);
    kern |= (p.cta2 ? kKernPair : 0) | (p.b_merged ? kKernBMerged : 0);
  }
  if (emitted_all && fuse.emitted) *fuse.emitted = true;
  note_conv(kPathTcBf16, kern);
  return true;
}

// ---- dgrad ---------------------------------------------------------------------------------------
static bool tc_conv_down_impl(const ConvGeom& g, const float* derivs, const float* filters, float* targets, float st, float so,
                              const Fuse& fuse, bool bf) {
  const Elem e = elem_for(bf);
  if (g.N % 4 != 0 || g.Cout % 4 != 0 || g.Cout < 8 || g.Cin < 8) return false;
  if (bf && (g.N % 8 != 0 || g.Cout % 8 != 0 || !aligned16(derivs) || !aligned16(filters))) return false;
  if (bf && (long long)g.N * g.W * g.H < 1024 && !bf16_staged(filters, (long long)g.Cout * g.K)) return false;   // see tc_conv_up_impl
  TcParams p; fill_common(p, g, e);
  p.BN = pick_bn(g.Cin, 16);
  p.kc_blocks = ceil_div(g.Cout, e.bk);
  const long long chunks = (long long)p.nb * g.W * g.H;
  if (chunks * 4 >= (1LL << 31) || g.kx > 32 || g.ky > 32) return false;
  p.total_chunks = p.nbc * g.W * g.H;
  p.m_tiles = ceil_div(p.total_chunks, p.cpt);
  p.n_tiles = ceil_div(g.Cin, p.BN);
  p.num_tiles = p.m_tiles * p.n_tiles;
  p.so = so;
  p.b_tx_bytes = (uint32_t)p.BN * 128;
  p.idesc = ptx::make_idesc(bf ? 1 : 2, true, false, BM, p.BN);
  const bool whole = (g.frames == 1 && g.cin0 == 0 && g.Cin == g.CinT);
  const long long out_elems = (long long)g.Cin * g.W * g.H * g.N;
  const int ks = whole ? pick_ksplit(p, g, out_elems) : 1;
  if (ks > 1) {
    p.units_per_split = ceil_div(p.kc_blocks, ks);
    p.splits = ceil_div(p.kc_blocks, p.units_per_split);
    p.part_stride = out_elems;
    p.num_tiles *= p.splits;
  }
  const size_t part_bytes = p.splits > 1 ? align_up(sizeof(float) * out_elems * p.splits) : 0;
  apply_pair(p, kDgrad, 8, 1);
  const int bn_local = p.cta2 ? p.BN / 2 : p.BN;
  CUtensorMap ma, mb;
  const long long der_off = (long long)g.cout0 * g.modules * g.N;
  const void* der = derivs + der_off;
  const void* flt = filters;
  uint8_t* ws = nullptr;
  if (bf) {
    const __nv_bfloat16* sd = bf16_staged(derivs, g.out_total);
    const __nv_bfloat16* sf = bf16_staged(filters, (long long)g.Cout * g.K);
    const size_t db = sd ? 0 : align_up((size_t)g.out_total * 2), fb = sf ? 0 : align_up((size_t)g.Cout * g.K * 2);
    if (part_bytes + db + fb) ws = (uint8_t*)workspace(part_bytes + db + fb);
    if (!sd) { to_bf16(derivs, (__nv_bfloat16*)(ws + part_bytes), g.out_total); sd = (const __nv_bfloat16*)(ws + part_bytes); }
    if (!sf) { to_bf16(filters, (__nv_bfloat16*)(ws + part_bytes + db), (long long)g.Cout * g.K); sf = (const __nv_bfloat16*)(ws + part_bytes + db); }
    der = sd + der_off;
    flt = sf;
  } else if (part_bytes) {
    ws = (uint8_t*)workspace(part_bytes);
  }
  p.a_merged = (allow_merge() && g.frames == 1 && g.N % 128 == 0) ? 1 : 0;
  if (p.a_merged) {
    if (!merged_image_map(&ma, der, e, g, g.modX, g.modY, g.Cout, false)) return false;
  } else if (!image_map(&ma, der, e, g, g.modX, g.modY, g.Cout, g.out_frame_step, true, e.bk)) return false;
  {
    const long long dims[3] = {g.Cout, (long long)g.kx * g.ky, g.Cin};
    const long long str[2] = {g.Cout, (long long)g.Cout * g.kx * g.ky};
    const int box[3] = {e.chunk, 1, bn_local};
    if (!make_map(&mb, flt, e, 3, dims, str, box, false)) return false;
  }
  float* out = targets + (long long)g.cin0 * g.H * g.W * g.N;
  if (whole && p.splits > 1) {
    p.st = 0.f; p.out = (float*)ws; p.mask = nullptr;
    launch<kDgrad>(ma, mb, p);
    reduce_split((const float*)ws, out, out_elems, p.splits, st, so, nullptr, 1, 0, fuse.relu_mask);
  } else if (whole) {
    p.st = st; p.out = out; p.mask = fuse.relu_mask ? fuse.relu_mask + (long long)g.cin0 * g.H * g.W * g.N : nullptr;
    p.out16 = fuse.out16;                              // `whole`: every element gets its final value here
    launch<kDgrad>(ma, mb, p);
    if (fuse.out16 && fuse.emitted) *fuse.emitted = true;
  } else {
    // the reference scales the WHOLE target first (gemm.cu:760, conv3d_gemm.cu:98); frame windows overlap,
    // so frames are accumulated by stream-ordered launches
    scale_buffer(targets, g.img_total, st);
    p.st = 1.f;
    for (int f = 0; f < g.frames; f++) {
      p.frame0 = f; p.out = out + f * g.in_frame_step;
      launch<kDgrad>(ma, mb, p);
    }
  }
  note_conv(bf ? kPathTcBf16 : kPathTcTf32,
            (p.cta2 ? kKernPair : 0) | (p.splits > 1 ? kKernSplit : 0) | (p.a_merged ? kKernAMerged : 0));
  return true;
}
bool tc_conv_down(const ConvGeom& g, const float* derivs, const float* filters, float* targets, float st, float so,
                  const Fuse& fuse) {
  if (!tc_enabled() || !g.conv) return false;
  if (want_bf16() && st == 0.f && tc_conv_down_as_fprop(g, derivs, filters, targets, so, fuse)) return true;
  if (want_bf16() && tc_conv_down_impl(g, derivs, filters, targets, st, so, fuse, true)) return true;
  return tc_conv_down_impl(g, derivs, filters, targets, st, so, fuse, false);
}

// ---- wgrad ---------------------------------------------------------------------------------------
static bool tc_conv_outp_impl(const ConvGeom& g, const float* images, const float* derivs, float* targets, float st, float so,
                              bool bf) {
  const Elem e = elem_for(bf);
  if (g.N % 4 != 0 || g.Cout < 8) return false;
  const bool x_mode = g.Cin < 8;
  if (x_mode && (g.kx > 8 || g.ky > 8)) return false;
  if (bf && (x_mode || g.N % 8 != 0 || !aligned16(images) || !aligned16(derivs))) return false;
  // few reduction rows (FC layers: K = batch): the call is bound by WRITING dW.  The general kernel gained nothing from bf16
  // there; the lean one (eight epilogue warps) does, and the operands it converts are tiny — so FC shapes take bf16 only when
  // they are eligible for it
  const bool lean_ok = fast_enabled() && !x_mode && g.frames == 1 && g.N % 128 == 0 && g.Cin % 32 == 0;
  if (bf && (long long)g.N * g.modules * g.frames < 1024 && !lean_ok) return false;
  TcParams p; fill_common(p, g, e);
  p.kc_blocks = 0;
  p.m_tiles = ceil_div(g.Cout, BM);
  if (x_mode) {
    p.x_mode = 1;
    p.x_ct = std::min(g.Cin, 256 / (8 * g.ky));      // channels per N tile: x_ct * ky * 8 columns
    p.BN = ceil_div(p.x_ct * g.ky * 8, 16) * 16;
    p.n_tiles = ceil_div(g.Cin, p.x_ct);
    p.b_tx_bytes = (uint32_t)p.x_ct * g.ky * 8 * 128;
  } else {
    p.BN = pick_bn(g.Cin, 16);
    p.n_tiles = ceil_div(g.Cin, p.BN);
    p.b_tx_bytes = (uint32_t)p.BN * 128;
  }
  const int units = g.modY * g.frames;               // reduction units = module rows
  const long long base_tiles = (long long)(x_mode ? 1 : p.taps) * p.m_tiles * p.n_tiles;
  // reduction splits: minimise  waves x (rows per tile x time of a row + epilogue)  +  the partial-sum reduction pass.
  // (The old rule — fill two waves — left e.g. 168 pair tiles for 74 pair slots.)  Times in microseconds, coarse: one
  // k-block ~0.3 us, a tile epilogue ~1.5 us, the reduction streams (splits + 1) x |dW| floats at ~5 TB/s.
  int splits;
  {
    const bool may_pair = pair_enabled() && !x_mode && p.m_tiles >= 2 && (p.m_tiles & 1) == 0;
    const long long slots = may_pair ? num_sms() / 2 : num_sms();
    const long long base = may_pair ? base_tiles / 2 : base_tiles;
    const double row_us = 0.3 * g.modX * std::max(1, p.nbc / 2);
    const double dw_bytes = 4.0 * g.Cout * g.K;
    const int cap = (int)std::max<long long>(1, std::min<long long>(units, (4LL * num_sms()) / std::max<long long>(base_tiles, 1)));
    double best = 1e30; splits = 1;
    for (int sp = 1; sp <= cap; sp++) {
      const int ups = ceil_div(units, sp), real = ceil_div(units, ups);
      const long long waves = ceil_div<long long>(base * real, slots);
      const double cost = (double)waves * (ups * row_us + 1.5) + (real > 1 ? dw_bytes * (real + 1) / 5e6 : 0.0);
      if (cost < best - 1e-9) { best = cost; splits = real; }
    }
  }
  const long long elems = (long long)g.Cout * g.K;
  while (splits > 1 && elems * splits * 4 > (1LL << 30)) splits--;
  p.units_per_split = ceil_div(units, splits);
  p.splits = ceil_div(units, p.units_per_split);
  p.num_tiles = (int)(base_tiles * p.splits);
  p.st = st; p.so = so;
  p.idesc = ptx::make_idesc(bf ? 1 : 2, false, false, BM, p.BN);
  apply_pair(p, kWgrad, 8, x_mode ? 1 : p.taps);
  const int bn_local = p.cta2 ? p.BN / 2 : p.BN;
  CUtensorMap ma, mb;
  const long long img_off = (long long)g.cin0 * g.H * g.W * g.N, der_off = (long long)g.cout0 * g.modules * g.N;
  const void* img = images + img_off;
  const void* der = derivs + der_off;
  const size_t part_bytes = p.splits > 1 ? align_up(sizeof(float) * elems * p.splits) : 0;
  uint8_t* ws = nullptr;
  if (bf) {
    const __nv_bfloat16* si = bf16_staged(images, g.img_total);
    const __nv_bfloat16* sd = bf16_staged(derivs, g.out_total);
    const size_t ib = si ? 0 : align_up((size_t)g.img_total * 2), db = sd ? 0 : align_up((size_t)g.out_total * 2);
    if (part_bytes + ib + db) ws = (uint8_t*)workspace(part_bytes + ib + db);
    if (!si) { to_bf16(images, (__nv_bfloat16*)(ws + part_bytes), g.img_total); si = (const __nv_bfloat16*)(ws + part_bytes); }
    if (!sd) { to_bf16(derivs, (__nv_bfloat16*)(ws + part_bytes + ib), g.out_total); sd = (const __nv_bfloat16*)(ws + part_bytes + ib); }
    img = si + img_off;
    der = sd + der_off;
  } else if (part_bytes) {
    ws = (uint8_t*)workspace(part_bytes);
  }
  if (!image_map(&ma, der, e, g, g.modX, g.modY, g.Cout, g.out_frame_step, false, BM)) return false;
  if (x_mode) {
    const long long N = g.N;
    const long long dims[5] = {N, g.W, g.H, g.Cin, g.frames};
    const long long str[4] = {N, N * g.W, N * g.W * g.H, g.in_frame_step};
    const int box[5] = {32, 8, g.ky, 1, 1};                   // 8 x-taps x ky rows of one channel: ky*8 GEMM columns
    if (!make_map(&mb, img, e, 5, dims, str, box, false)) return false;
  } else if (!image_map(&mb, img, e, g, g.W, g.H, g.Cin, g.in_frame_step, false, bn_local)) return false;
  p.out = p.splits == 1 ? targets : (float*)ws;
  bool done = false;
  int kern = (p.cta2 ? kKernPair : 0) | (x_mode ? kKernXMode : 0) | (p.splits > 1 ? kKernSplit : 0);
  if (bf && fast_enabled() && !x_mode && g.frames == 1 && g.N % 128 == 0 && g.Cin % 32 == 0 && p.BN % 32 == 0 &&
      (p.splits > 1 || st == 0.f)) {
    TcParams f = p;
    if (p.splits > 1) f.so = 1.f;                      // partial sums are scaled by reduce_partials
    if (fast_pick_stages(f, bn_local)) {
      const long long N = g.N, cps = f.ksteps / 4;
      // (n_lo = 64, x, y, channel, n_hi = N/64) views: one request brings `cps` 64-image panels of a module
      const long long adims[5] = {64, g.modX, g.modY, g.Cout, N / 64}, astr[4] = {N, N * g.modX, N * g.modX * g.modY, 64};
      const int abox[5] = {64, 1, 1, BM, (int)cps};
      const long long bdims[5] = {64, g.W, g.H, g.Cin, N / 64}, bstr[4] = {N, N * g.W, N * g.W * g.H, 64};
      const int bbox[5] = {64, 1, 1, bn_local, (int)cps};
      CUtensorMap fa, fb;
      if (make_map(&fa, der, e, 5, adims, astr, abox, false) && make_map(&fb, img, e, 5, bdims, bstr, bbox, false)) {
        launch_fast<kWgrad>(fa, fb, f);
        done = true;
        kern |= kKernLean;
      }
    }
  }
  if (!done && !bf && x_mode && fast_enabled() && g.frames == 1 && g.N % 64 == 0 && !p.cta2 && (p.splits > 1 || st == 0.f)) {
    TcParams f = p;
    if (p.splits > 1) f.so = 1.f;
    const int cps = 2, rows_panel = p.x_ct * g.ky * 8;             // 64 images per stage; tap rows of one 32-image panel
    f.ksteps = 4 * cps; f.a_stage_bytes = 16384u * cps;
    f.b_rows = rows_panel * cps + 8;                               // the MMA reads BN >= rows_panel rows of the last panel
    f.b_tx_bytes = (uint32_t)(rows_panel * cps) * 128;
    int stages = kMaxStages;
    while (stages > 1 && fast_smem_bytes(f.a_stage_bytes, (size_t)f.b_rows * 128, stages) > 225 * 1024) stages--;
    f.stages = stages;
    const long long N = g.N;
    const long long adims[5] = {32, g.modX, g.modY, g.Cout, N / 32}, astr[4] = {N, N * g.modX, N * g.modX * g.modY, 32};
    const int abox[5] = {32, 1, 1, BM, cps};
    const long long bdims[5] = {32, g.W, g.H, g.Cin, N / 32}, bstr[4] = {N, N * g.W, N * g.W * g.H, 32};
    const int bbox[5] = {32, 8, g.ky, p.x_ct, cps};
    CUtensorMap fa, fb;
    if (stages >= 2 && make_map(&fa, der, e, 5, adims, astr, abox, false) && make_map(&fb, img, e, 5, bdims, bstr, bbox, false)) {
      launch_fast<kWgrad, true>(fa, fb, f);
      done = true;
      kern |= kKernLean;
    }
  }
  if (!done) launch<kWgrad>(ma, mb, p);
  if (p.splits > 1) reduce_partials((const float*)ws, targets, elems, 1, p.splits, st, so);
  note_conv(bf ? kPathTcBf16 : kPathTcTf32, kern);
  return true;
}
bool tc_conv_outp(const ConvGeom& g, const float* images, const float* derivs, float* targets, float st, float so) {
  if (!tc_enabled() || !g.conv) return false;
  if (want_bf16() && tc_conv_outp_impl(g, images, derivs, targets, st, so, true)) return true;
  return tc_conv_outp_impl(g, images, derivs, targets, st, so, false);
}

}  // namespace cnb
