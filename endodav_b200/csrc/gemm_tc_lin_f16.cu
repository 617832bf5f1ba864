// tcgen05 linear GEMMs, f16 operands (one translation unit per (dtype, lin|conv) slice: parallel nvcc)
#define EDV_GEMM_TU_LIN
#define EDV_GEMM_TU_LN   // this TU also holds the non-template gemm_ln() dispatcher (both dtypes)
#include "gemm_tc_inst.cuh"
namespace edv { template void launch_gemm_tc_lin<f16>(Launch&, int, const GemmArgs&); }
