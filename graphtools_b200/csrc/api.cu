// Error reporting + version for libgtb200.so
#include "common.cuh"
#include "gtb200.h"
#include <stdarg.h>

static thread_local char g_err[512] = "";

void gtb_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

extern "C" const char* gtb_last_error(void) { return g_err; }
extern "C" int gtb_version(void) { return 206; }   // + gtb_spmm_cheb_acc, gtb_laplacian_count/_fill (csrc/gsp.cu)
