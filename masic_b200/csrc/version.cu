// version.cu — ABI version / build string of libmasic_b200.so
#include "../../include/masic_b200.h"
#define MASIC_STR2(x) #x
#define MASIC_STR(x) MASIC_STR2(x)
extern "C" int masic_abi_version(void) { return 11; }
extern "C" const char* masic_build_info(void) {
  return "masic_b200 sm_100a nvcc " MASIC_STR(__CUDACC_VER_MAJOR__) "." MASIC_STR(__CUDACC_VER_MINOR__)
         " (tcgen05+TMA implicit-GEMM convs, fused entropy/warp kernels)";
}
