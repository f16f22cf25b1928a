// capi.cu -- library-level pieces of the C ABI: version, status strings, thread-local error
// detail, and the reference's thread-count rule.
#include <math.h>
#include <stdarg.h>

#include "common.cuh"

namespace b2r {
namespace {
thread_local char g_err[512] = "";
}
void set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
}  // namespace b2r

extern "C" int b2r_version(void) { return 100; /* 0.1.0 */ }

extern "C" const char *b2r_status_string(int status) {
  switch (status) {
    case B2R_OK: return "ok";
    case B2R_ERR_INVALID_ARG: return "invalid argument";
    case B2R_ERR_CUDA: return "CUDA error";
    case B2R_ERR_UNSUPPORTED: return "unsupported size";
    default: return "unknown status";
  }
}

extern "C" const char *b2r_last_error(void) { return b2r::g_err; }

extern "C" int b2r_struct_bytes(int which) {
  if (which == 0) return (int)sizeof(b2r_sa_layer);
  if (which == 1) return (int)sizeof(b2r_sa_layer_bwd_desc);
  if (which == 2) return (int)sizeof(b2r_dense_layer);
  if (which == 3) return (int)sizeof(b2r_dense_layer_bwd);
  if (which == 4) return (int)sizeof(b2r_adam_desc);
  return -1;
}

// Reference include/cuda_utils.h:20-24 (opt_n_threads): 2^floor(log2(work)) capped to [1,512],
// computed with the same double log()/log(2.0) quotient and int truncation so that the FPS tie
// order (which depends on this value) matches on every N, including exact powers of two.
extern "C" int b2r_ref_block_threads(int work_size) {
  if (work_size < 1) return 1;
  const int p = (int)(log((double)work_size) / log(2.0));
  int t = 1 << p;
  if (t > 512) t = 512;
  if (t < 1) t = 1;
  return t;
}
