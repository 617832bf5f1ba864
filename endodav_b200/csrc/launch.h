// Launch bookkeeping shared by all host-side launchers.
#pragma once
#include <cuda_runtime.h>

#include <cstdlib>
#include <string>
#include <utility>
#include <vector>

#include "../../include/endodav_b200.h"

namespace edv {

// EDV_PDL=0 launches every kernel fully serialised (no programmatic dependent launch)
inline bool pdl_enabled() {
  static const bool v = [] { const char* e = getenv("EDV_PDL"); return !e || atoi(e) != 0; }();
  return v;
}

// kern<<<grid, block, smem, stream>>>(args...) with programmatic stream serialisation: the kernel may be scheduled
// while its predecessor in the stream is still running and must call pdl_wait() (common.cuh) before touching global
// memory.  Works under stream capture (programmatic edges in the captured graph).
template <typename... KArgs, typename... Args>
inline void launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

// Allows kernel Kern up to `bytes` of dynamic shared memory; sets the attribute on the first call only, so eager
// forwards pay no host time for it.  The kernel itself is the template argument: a flag in a helper templated on the
// kernel's signature would be shared by all instances of a kernel template (e.g. every gemm_tc_kernel<T, BN, BK, CONV>).
template <auto Kern> inline void smem_opt_in(int bytes) {
  static bool done = false;
  if (!done) {
    cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    done = true;
  }
}

// Optional per-launch timing: one CUDA event after every launch on the launching stream, so
// the duration of launch i is event[i] - event[i-1] (the stream is serial).  Used by bench.py
// for the live roofline numbers; off by default (no events are recorded).
struct ProfRec {
  std::string name;   // "" marks the start of a forward
  double flops, bytes;
};
struct Profiler {
  bool on = false;
  std::vector<cudaEvent_t> ev;
  std::vector<ProfRec> recs;
  size_t used = 0;
  cudaEvent_t next() {
    if (used == ev.size()) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      ev.push_back(e);
    }
    return ev[used++];
  }
  void mark(cudaStream_t s, const std::string& name, double flops, double bytes) {
    cudaEventRecord(next(), s);
    recs.push_back(ProfRec{name, flops, bytes});
  }
  ~Profiler() {
    for (cudaEvent_t e : ev) cudaEventDestroy(e);
  }
};

struct Launch {
  cudaStream_t stream = nullptr;
  int count = 0;         // kernels launched
  int status = EDV_OK;   // first error
  std::string err;
  Profiler* prof = nullptr;
  std::string tag;       // which call site of the forward graph the next launches belong to
  std::string kernel;    // the GEMM, attention or head instance launched last, e.g. "gemm_tc<BN=32,BK=64,kind=0x9,tma=0>",
                         // "temporal_attention_mma<HD=24,PB=2>", "flash_attention_tc<bf16>", "head_fused<bf16,CIN=128>"
                         // (edv_op_gemm, edv_op_temporal_attention, edv_op_attention, edv_op_disp_head)
  double nflops = 0, nbytes = 0;  // algorithmic work of the next launch (set by the launcher)

  void note(double flops, double bytes) {
    nflops = flops;
    nbytes = bytes;
  }
  void begin() {
    if (prof && prof->on) prof->mark(stream, "", 0, 0);
  }

  void fail(int code, const std::string& what) {
    if (status == EDV_OK) {
      status = code;
      err = what;
    }
  }
  void check(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) fail(EDV_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
    ++count;
    if (prof && prof->on) prof->mark(stream, tag.empty() ? std::string(what) : std::string(what) + ":" + tag, nflops, nbytes);
    nflops = nbytes = 0;
  }
  bool ok() const { return status == EDV_OK; }
};

}  // namespace edv
