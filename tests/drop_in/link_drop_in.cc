// link_drop_in.cc — link-level drop-in proof (TEST INFRASTRUCTURE).
//
// This translation unit includes the REFERENCE'S OWN headers, cudamat/cudamat_conv_gemm.cuh and
// cudamat/cudamat_conv.cuh (-I$REF/cudamat at compile time; nothing of them is copied here), declares nothing
// itself, and is linked with `-lcudamat_conv_gemm -lcudamat_conv` resolved from convnet_b200/lib — the two library
// names the reference's Makefile:72-77 links.  If a prototype, a struct layout or a symbol name of the product
// differed from the reference's, this file would fail to compile, to link, or to compute the right numbers.
// Without the reference's headers (DROP_IN_OWN_HEADERS) it includes the project's declarations of the same two ABIs,
// and still proves the library names, both symbol sets and the numbers.  Built by convnet_b200/build.py build_drop_in.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>

#ifdef DROP_IN_OWN_HEADERS
#include "convnet_b200_conv_gemm.h"
#include "convnet_b200_conv.h"
#else
#include "cudamat_conv_gemm.cuh"   // the reference's ABI-1 header (pulls in cudamat.cuh: cudamat, Shape4D, ConvDesc)
#include "cudamat_conv.cuh"        // the reference's ABI-2 header
#endif

static void ck(cudaError_t e, const char* what) {
  if (e != cudaSuccess) { fprintf(stderr, "%s: %s\n", what, cudaGetErrorString(e)); exit(2); }
}

struct DevMat {
  cudamat m;
  Shape4D s;
  std::vector<float> h;
  DevMat(int rows, int cols, int a, int b, int c, int d) : h((size_t)rows * cols, 0.f) {
    m.data_host = nullptr; m.on_device = 1; m.on_host = 0; m.size[0] = rows; m.size[1] = cols;
    m.is_trans = 0; m.owns_data = 1; m.tex_obj = 0;
    ck(cudaMalloc((void**)&m.data_device, sizeof(float) * h.size()), "cudaMalloc");
    s.shape[0] = a; s.shape[1] = b; s.shape[2] = c; s.shape[3] = d;
  }
  ~DevMat() { cudaFree(m.data_device); }
  void up() { ck(cudaMemcpy(m.data_device, h.data(), sizeof(float) * h.size(), cudaMemcpyHostToDevice), "H2D"); }
  void down() { ck(cudaMemcpy(h.data(), m.data_device, sizeof(float) * h.size(), cudaMemcpyDeviceToHost), "D2H"); }
};

static float frand(unsigned& s) { s = s * 1664525u + 1013904223u; return ((s >> 8) & 0xFFFF) / 32768.0f - 1.0f; }

static double rel_diff(const std::vector<float>& a, const std::vector<double>& b) {
  double mx = 0, mean = 0;
  for (size_t i = 0; i < a.size(); i++) { mx = std::fmax(mx, std::fabs(a[i] - b[i])); mean += std::fabs(a[i] + b[i]); }
  return mx / (mean / a.size());
}

int main() {
  setenv("CONVNET_B200_PRECISION", "fp32", 1);     // product extension (read once); harmless for any other library
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { fprintf(stderr, "no CUDA device\n"); return 3; }
  const int N = 32, W = 6, H = 6, Cin = 8, Cout = 16, k = 3, pad = 1;
  ConvDesc d;
  d.num_input_channels = Cin; d.num_output_channels = Cout;
  d.kernel_size_y = d.kernel_size_x = k; d.kernel_size_t = 1;
  d.stride_y = d.stride_x = d.stride_t = 1;
  d.padding_y = d.padding_x = -pad; d.padding_t = 0;          // negated, src/edge.cc:97-99
  d.input_channel_begin = 0; d.input_channel_end = Cin; d.output_channel_begin = 0; d.output_channel_end = Cout;
  d.num_groups = 1;
  DevMat img(N, W * H * Cin, N, W, H, Cin), flt(Cout, k * k * Cin, Cout, k, k, Cin);
  DevMat out1(N, W * H * Cout, N, W, H, Cout), out2(N, W * H * Cout, N, W, H, Cout);
  unsigned seed = 7;
  for (float& v : img.h) v = frand(seed);
  for (float& v : flt.h) v = frand(seed) * 0.2f;
  img.up(); flt.up();
  // CPU brute force from the index formulas of SURVEY.md Appendix A
  std::vector<double> ref((size_t)N * W * H * Cout, 0.0);
  for (int o = 0; o < Cout; o++)
    for (int my = 0; my < H; my++)
      for (int mx = 0; mx < W; mx++)
        for (int n = 0; n < N; n++) {
          double acc = 0;
          for (int c = 0; c < Cin; c++)
            for (int ty = 0; ty < k; ty++)
              for (int tx = 0; tx < k; tx++) {
                const int y = my - pad + ty, x = mx - pad + tx;
                if (x < 0 || x >= W || y < 0 || y >= H) continue;
                acc += (double)img.h[n + (size_t)N * (x + W * (y + H * c))] * flt.h[o + (size_t)Cout * (tx + k * (ty + k * c))];
              }
          ref[n + (size_t)N * (mx + W * (my + H * o))] = acc;
        }
  convUpGemm(&img.m, &flt.m, &out1.m, &img.s, &flt.s, &out1.s, d, 0.f);       // ABI-1
  SetupTexture(&img.m);
  convUp(&img.m, &flt.m, &out2.m, &img.s, &flt.s, &out2.s, d, 0.f);           // ABI-2
  ck(cudaDeviceSynchronize(), "sync");
  out1.down(); out2.down();
  const double d1 = rel_diff(out1.h, ref), d2 = rel_diff(out2.h, ref);
  printf("convUpGemm Diff %.3e   convUp Diff %.3e\n", d1, d2);
  if (!(d1 < 1e-4) || !(d2 < 1e-4)) return 1;

  // 3x3 stride-2 max-pool through both symbol sets
  ConvDesc p = d;
  p.num_input_channels = p.num_output_channels = Cin; p.input_channel_end = p.output_channel_end = Cin;
  p.stride_y = p.stride_x = 2;
  const int mod = (W + 2 * pad - k) / 2 + 1;
  DevMat pool1(N, mod * mod * Cin, N, mod, mod, Cin), pool2(N, mod * mod * Cin, N, mod, mod, Cin);
  MaxPoolGemm(&img.m, &pool1.m, &img.s, &pool1.s, p, 0.f, 1.f);
  MaxPool(&img.m, &pool2.m, &img.s, &pool2.s, p);
  ck(cudaDeviceSynchronize(), "sync");
  pool1.down(); pool2.down();
  for (int c = 0; c < Cin; c++)
    for (int my = 0; my < mod; my++)
      for (int mx = 0; mx < mod; mx++)
        for (int n = 0; n < N; n++) {
          float best = -2e38f;
          for (int ty = 0; ty < k; ty++)
            for (int tx = 0; tx < k; tx++) {
              const int y = my * 2 - pad + ty, x = mx * 2 - pad + tx;
              if (x < 0 || x >= W || y < 0 || y >= H) continue;
              best = std::fmax(best, img.h[n + (size_t)N * (x + W * (y + H * c))]);
            }
          const size_t i = n + (size_t)N * (mx + mod * (my + mod * c));
          if (pool1.h[i] != best || pool2.h[i] != best) { printf("max-pool mismatch at %zu\n", i); return 1; }
        }
  printf("MaxPoolGemm / MaxPool bit-exact\nDROP-IN OK\n");
  return 0;
}
