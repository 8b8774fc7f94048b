// abi_facts.cc — what a set of headers declares for the two reference symbol sets (TEST INFRASTRUCTURE).
//
// Prints, for every function of both symbol sets, the compiler's name of its type (Itanium ABI: return and parameter
// types), and the sizes of the three ABI structs.  Taking every function's address makes each one an undefined symbol
// of the linked binary, under the linkage its declaration gives it.  Compiled against the reference's own headers
// (cudamat/cudamat_conv_gemm.cuh, cudamat/cudamat_conv.cuh) and against the project's (DROP_IN_OWN_HEADERS), the two
// outputs and symbol lists must be identical: tests/test_link_drop_in.py, which stores the reference's side.
#include <cstdio>
#include <typeinfo>

#ifdef DROP_IN_OWN_HEADERS
#include "convnet_b200_conv_gemm.h"
#include "convnet_b200_conv.h"
#else
#include "cudamat_conv_gemm.cuh"
#include "cudamat_conv.cuh"
#endif

#define ABI_FUNCTIONS(X)                                                                                              \
  X(convUpGemm) X(convDownGemm) X(convOutpGemm) X(convInnerpGemm) X(localUpGemm) X(localDownGemm) X(localOutpGemm)    \
  X(MaxPoolGemm) X(MaxPoolUndoGemm) X(MaxPoolRpropGemm) X(AvgPoolGemm) X(AvgPoolUndoGemm) X(UpSampleGemm)              \
  X(DownSampleGemm) X(ResponseNormCrossMapGemm) X(ResponseNormCrossMapUndoGemm) X(ResponseNormCrossMapRpropGemm)       \
  X(Scale) X(convUp3DGemm) X(convDown3DGemm) X(convOutp3DGemm) X(ResponseNormCrossMap3DGemm)                           \
  X(ResponseNormCrossMap3DUndoGemm)                                                                                    \
  X(SetupTexture) X(convUp) X(localUp) X(convDown) X(localDown) X(convOutp) X(localOutp) X(ResponseNormCrossMap)       \
  X(ResponseNormCrossMapUndo) X(ResponseNorm) X(ResponseNormUndo) X(ContrastNorm) X(ContrastNormUndo) X(MaxPool)       \
  X(AvgPool) X(MaxPoolUndo) X(AvgPoolUndo) X(UpSample) X(DownSample) X(RGBToYUV)

#define ADDRESS(f) reinterpret_cast<void*>(&f),
void* volatile keep[] = {ABI_FUNCTIONS(ADDRESS)};

int main() {
#define PRINT(f) printf("%s %s\n", #f, typeid(decltype(f)).name());
  ABI_FUNCTIONS(PRINT)
  printf("sizeof(cudamat) %zu\nsizeof(Shape4D) %zu\nsizeof(ConvDesc) %zu\n", sizeof(cudamat), sizeof(Shape4D),
         sizeof(ConvDesc));
  return keep[0] == nullptr;
}
