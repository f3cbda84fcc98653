// Library-level entry points of the C ABI (include/ic3net_b200.h).
#include "ic3_common.cuh"

unsigned long long g_ic3_launches = 0;

extern "C" const char* ic3_version(void) { return "ic3net_b200 0.1 (sm_100a)"; }

extern "C" uint64_t ic3_launch_count(void) { return (uint64_t)g_ic3_launches; }

extern "C" const char* ic3_strerror(int code) {
  switch (code) {
    case IC3_OK: return "ok";
    case IC3_E_NULL: return "required pointer is NULL";
    case IC3_E_RANGE: return "argument out of the supported range";
    case IC3_E_UNSUPPORTED: return "configuration not implemented by the kernels";
    default: break;
  }
  if (code > 0) return cudaGetErrorString((cudaError_t)code);
  return "unknown ic3 error";
}
