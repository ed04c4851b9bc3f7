// api.cu — C-ABI glue: versioning, error strings, and the conv dispatcher (tensor-core path vs exact SIMT path).
#include "common.cuh"

int g_dp_last_cuda_error = 0;
long long g_dp_launch_count = 0;

int dp_conv2d_fprop_simt(const dp_conv_args*, dp_stream_t);
int dp_conv2d_dgrad_simt(const dp_conv_args*, dp_stream_t);
int dp_conv2d_wgrad_simt(const dp_conv_args*, dp_stream_t);
#ifdef DPB200_HAVE_TC
int dp_conv2d_fprop_tc(const dp_conv_args*, dp_stream_t);   // returns DP_ERR_UNSUPPORTED when the shape is not eligible
int dp_conv2d_dgrad_tc(const dp_conv_args*, dp_stream_t);
int dp_conv2d_wgrad_tc(const dp_conv_args*, dp_stream_t);
int dp_tc_runtime_ok();
#endif

extern "C" int dp_version(void) { return 100; }  // 0.1.0

extern "C" const char* dp_strerror(int code) {
  switch (code) {
    case DP_OK: return "ok";
    case DP_ERR_SHAPE: return "inconsistent or out-of-range extents";
    case DP_ERR_ALIGN: return "pointer/stride alignment not supported by the kernel";
    case DP_ERR_UNSUPPORTED: return "request outside the implemented set";
    case DP_ERR_CUDA: return "CUDA launch failed (see dp_last_cuda_error)";
    case DP_ERR_NULL: return "required pointer is NULL";
    default: return "unknown dpb200 error";
  }
}
extern "C" int dp_last_cuda_error(void) { return g_dp_last_cuda_error; }
extern "C" int64_t dp_launch_count(void) { return g_dp_launch_count; }

extern "C" int dp_tc_available(void) {
#ifdef DPB200_HAVE_TC
  return dp_tc_runtime_ok();
#else
  return 0;
#endif
}

// DP_CONV_X_SPLIT (an operand only the tensor-core kernels read) never falls back to the SIMT path
extern "C" int dp_conv2d_fprop(const dp_conv_args* a, dp_stream_t s) {
#ifdef DPB200_HAVE_TC
  if (a && !(a->flags & DP_CONV_FORCE_SIMT)) {
    int rc = dp_conv2d_fprop_tc(a, s);
    if (rc != DP_ERR_UNSUPPORTED || (a->flags & DP_CONV_X_SPLIT)) return rc;
  }
#endif
  if (a && (a->flags & DP_CONV_X_SPLIT)) return DP_ERR_UNSUPPORTED;
  return dp_conv2d_fprop_simt(a, s);
}
extern "C" int dp_conv2d_dgrad(const dp_conv_args* a, dp_stream_t s) {
#ifdef DPB200_HAVE_TC
  if (a && !(a->flags & DP_CONV_FORCE_SIMT)) {
    int rc = dp_conv2d_dgrad_tc(a, s);
    if (rc != DP_ERR_UNSUPPORTED) return rc;
  }
#endif
  return dp_conv2d_dgrad_simt(a, s);
}
extern "C" int dp_conv2d_wgrad(const dp_conv_args* a, dp_stream_t s) {
#ifdef DPB200_HAVE_TC
  if (a && !(a->flags & DP_CONV_FORCE_SIMT)) {
    int rc = dp_conv2d_wgrad_tc(a, s);
    if (rc != DP_ERR_UNSUPPORTED || (a->flags & DP_CONV_X_SPLIT)) return rc;
  }
#endif
  if (a && (a->flags & DP_CONV_X_SPLIT)) return DP_ERR_UNSUPPORTED;
  return dp_conv2d_wgrad_simt(a, s);
}
