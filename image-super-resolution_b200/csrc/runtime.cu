// Error reporting and device gate of libffsr_b200.so.
#include "common.cuh"
#include <stdarg.h>
#include <stdio.h>
#include "../../include/ffsr_b200.h"

static thread_local char g_err[512] = "";

void ffsr_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int ffsr_check_launch(const char* what) {
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    ffsr_set_error("%s: launch failed: %s", what, cudaGetErrorString(e));
    return FFSR_ERR_LAUNCH;
  }
  return FFSR_OK;
}

extern "C" const char* ffsr_last_error(void) { return g_err; }
extern "C" const char* ffsr_version(void) { return "ffsr_b200 0.5 (sm_100a)"; }

// The library carries sm_100a SASS only: refuse anything else loudly instead of falling back.
extern "C" int ffsr_device_check(void) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    ffsr_set_error("device_check: no CUDA device: %s", cudaGetErrorString(e));
    return FFSR_ERR_DRIVER;
  }
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, dev);
  if (e != cudaSuccess) {
    ffsr_set_error("device_check: %s", cudaGetErrorString(e));
    return FFSR_ERR_DRIVER;
  }
  if (prop.major != 10) {
    ffsr_set_error("device_check: %s is sm_%d%d; libffsr_b200 is built for sm_100a (B200) only", prop.name, prop.major,
                   prop.minor);
    return FFSR_ERR_ARG;
  }
  return FFSR_OK;
}

// lets a binding verify its struct layout against the library it loaded
extern "C" size_t ffsr_conv_params_size(void) { return sizeof(ffsr_conv_params); }
