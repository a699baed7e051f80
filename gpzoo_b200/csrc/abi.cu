// ABI version and error strings.
#include "common.cuh"
#include "gpzoo_b200.h"

// 2: kernel_build_* take `kind`; 3: sparse-count K7 (poisson_*_csc_*); 4: the separate Cholesky and triangular-inverse entry
// points are gone (gpz_chol_inv_* computes both), gpz_svgp_predict_bwd_h_f32 lost its Lc argument
extern "C" int gpz_abi_version(void) { return 4; }

extern "C" const char* gpz_error_string(int rc) {
  if (rc == 0) return "success";
  if (rc == GPZ_ERR_BADARG) return "gpzoo_b200: bad argument";
  if (rc == GPZ_ERR_UNSUPPORTED) return "gpzoo_b200: unsupported size (see limits in csrc/*.cu)";
  if (rc < 0 && rc > -1000) return cudaGetErrorString((cudaError_t)(-rc));
  return "gpzoo_b200: unknown error";
}

#include <atomic>
static std::atomic<long long> g_launches{0};
extern "C" void gpz_count_launch_(void) { g_launches.fetch_add(1, std::memory_order_relaxed); }
// number of CUDA kernels this library has launched in this process (bench.py "gpu_launches")
extern "C" long long gpz_launch_count(void) { return g_launches.load(); }
