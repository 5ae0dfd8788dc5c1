// C-ABI plumbing: error reporting and dispatch between the arithmetic arms.
#include <cstdarg>
#include <cstdio>
#include "common.cuh"
#include "../../include/demucs_b200.h"

static thread_local char g_err[512] = "";

void bd_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int bd_check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    bd_set_error("%s: launch failed: %s", what, cudaGetErrorString(e));
    return BD_ERR_CUDA;
  }
  return BD_OK;
}

int bd_conv_gemm_simt(const bd_gemm_desc* d, void* stream);
int bd_conv_gemm_tc(const bd_gemm_desc* d, void* stream, int* handled);
bool bd_conv_gemm_tc_eligible(const bd_gemm_desc& d);
int bd_conv_gemm_tc_tile(const bd_gemm_desc& d);
int bd_attention_simt(const float* q, const float* k, const float* v, float* o, int B, int H, int Tq, int Tk, int ldq,
                      int ldk, int ldv, int ldo, void* stream);
int bd_attention_tc(const float* q, const float* k, const float* v, float* o, int B, int H, int Tq, int Tk, int ldq,
                    int ldk, int ldv, int ldo, int math, float* ws, void* stream);
long long bd_attention_ws_floats(int B, int H, int Tq, int Tk, int math);
int bd_attention_b16(const float* q, const float* k, const float* v, float* o, int B, int H, int Tq, int Tk, int ldq,
                     int ldk, int ldv, int ldo, int math, float* ws, void* stream);
long long bd_attention_b16_ws_floats(int B, int H, int Tq, int Tk, int math);

extern "C" {

const char* bd_last_error(void) { return g_err; }
int bd_version(void) { return 4; }   // 4: bd_pcm_decode (WAV input decoded on the device); 3: bf16-operand arithmetic, gather / PCM entry points

int bd_conv_gemm(const bd_gemm_desc* d, void* stream) {
  if (!d) {
    bd_set_error("bd_conv_gemm: null descriptor");
    return BD_ERR_ARG;
  }
  if (d->math != BD_MATH_FP32) {
    int handled = 0;
    int rc = bd_conv_gemm_tc(d, stream, &handled);
    if (rc != BD_OK || handled) return rc;
  }
  if (d->x_bf16 || d->out_bf16) {
    bd_set_error("bd_conv_gemm: bf16 tensors need the tensor-core arm (BD_MATH_BF16, Cin %% 64 == 0, N >= 16, M >= 128)");
    return BD_ERR_ARG;
  }
  return bd_conv_gemm_simt(d, stream);
}

int bd_conv_gemm_arm(const bd_gemm_desc* d) {
  return (d && d->math != BD_MATH_FP32) ? bd_conv_gemm_tc_tile(*d) : 0;
}

int bd_attention(const float* q, const float* k, const float* v, float* o, int B, int H, int Tq, int Tk, int ldq,
                 int ldk, int ldv, int ldo, int math, float* ws, void* stream) {
  if (math == BD_MATH_TF32 || math == BD_MATH_TF32X3)
    return bd_attention_tc(q, k, v, o, B, H, Tq, Tk, ldq, ldk, ldv, ldo, math, ws, stream);
  if (math == BD_MATH_BF16X3 || math == BD_MATH_BF16)
    return bd_attention_b16(q, k, v, o, B, H, Tq, Tk, ldq, ldk, ldv, ldo, math, ws, stream);
  return bd_attention_simt(q, k, v, o, B, H, Tq, Tk, ldq, ldk, ldv, ldo, stream);
}

long long bd_attention_workspace(int B, int H, int Tq, int Tk, int math) {
  if (math == BD_MATH_BF16X3 || math == BD_MATH_BF16) return bd_attention_b16_ws_floats(B, H, Tq, Tk, math);
  if (math != BD_MATH_TF32 && math != BD_MATH_TF32X3) return 0;
  return bd_attention_ws_floats(B, H, Tq, Tk, math);
}

}  // extern "C"
