// C ABI glue: error reporting and the low-level op entry points used by the unit tests.
#include <string>

#include "../../include/diarizen_b200.h"
#include "common.cuh"
#include "gemm.h"
#include "seg_kernels.h"

namespace dz {
std::string& tls_error() {
  static thread_local std::string e;
  return e;
}
int fail(int code, const std::string& msg) {
  tls_error() = msg;
  return code;
}
int relpos_bucket(int d);
}  // namespace dz

using namespace dz;

extern "C" {

const char* dz_last_error(void) { return tls_error().c_str(); }
int dz_abi_version(void) { return 1; }

int dz_relpos_bucket(int d) { return relpos_bucket(d); }

int dz_gemm(const dz_gemm_desc* d, int impl, int force_bn, void* stream) {
  if (!d) return fail(DZ_ERR_INVALID, "null descriptor");
  cudaStream_t st = (cudaStream_t)stream;
  if (impl == 1) {
    cudaError_t e = gemm_simt_launch(*d, st);
    return e == cudaSuccess ? DZ_OK : fail(DZ_ERR_CUDA, cudaGetErrorString(e));
  }
  GemmPlan* p = gemm_plan_create(*d, force_bn);
  if (!p) return fail(DZ_ERR_CUDA, gemm_last_error());
  cudaError_t e = gemm_plan_launch(p, st);
  gemm_plan_destroy(p);  // tensor maps are passed by value at launch
  return e == cudaSuccess ? DZ_OK : fail(DZ_ERR_CUDA, cudaGetErrorString(e));
}

dz_gemm_plan* dz_gemm_plan_create(const dz_gemm_desc* d, int force_bn) {
  if (!d) { fail(DZ_ERR_INVALID, "null descriptor"); return nullptr; }
  GemmPlan* p = gemm_plan_create(*d, force_bn);
  if (!p) fail(DZ_ERR_CUDA, gemm_last_error());
  return reinterpret_cast<dz_gemm_plan*>(p);
}
int dz_gemm_plan_launch(const dz_gemm_plan* p, void* stream) {
  if (!p) return fail(DZ_ERR_INVALID, "null plan");
  cudaError_t e = gemm_plan_launch(reinterpret_cast<const GemmPlan*>(p), (cudaStream_t)stream);
  return e == cudaSuccess ? DZ_OK : fail(DZ_ERR_CUDA, cudaGetErrorString(e));
}
void dz_gemm_plan_destroy(dz_gemm_plan* p) { gemm_plan_destroy(reinterpret_cast<GemmPlan*>(p)); }

int dz_layernorm(const float* x_dev, int64_t rows, int C, int ldx, const float* prescale_dev, const float* gamma_dev,
                 const float* beta_dev, int act, float* y_f32_dev, int ldy, void* y_bf_dev, int64_t bf_plane, int ldb,
                 int planes, float* mix_dev, float mix_w, int mix_src, int mix_init, int fp16, void* stream) {
  // both kernels move rows in 16-byte float4 chunks (x, y_f32, mix) and 8-byte 16-bit chunks (y_bf), so every row
  // start has to stay aligned; they also hold at most 1024 columns in registers
  if (!x_dev || !gamma_dev || !beta_dev || rows < 1) return fail(DZ_ERR_INVALID, "layernorm: null pointer or no rows");
  if (C < 1 || C > 1024) return fail(DZ_ERR_INVALID, "layernorm: C must be in [1, 1024]");
  if (ldx < C || ldx % 4 != 0) return fail(DZ_ERR_INVALID, "layernorm: ldx must be >= C and a multiple of 4");
  if (y_f32_dev && (ldy < C || ldy % 4 != 0)) return fail(DZ_ERR_INVALID, "layernorm: ldy must be >= C and a multiple of 4");
  if (y_bf_dev && (ldb < C || ldb % 8 != 0 || bf_plane % 8 != 0 || (planes != 1 && planes != 2)))
    return fail(DZ_ERR_INVALID, "layernorm: ldb must be >= C, ldb and bf_plane multiples of 8, planes 1 or 2");
  if (act < 0 || act > 3) return fail(DZ_ERR_INVALID, "layernorm: act must be 0..3");
  if (mix_dev && mix_src != 1 && mix_src != 2) return fail(DZ_ERR_INVALID, "layernorm: mix_src must be 1 or 2");
  LnArgs a{};
  a.x = x_dev; a.rows = rows; a.C = C; a.ldx = ldx; a.prescale = prescale_dev; a.gamma = gamma_dev; a.beta = beta_dev;
  a.act = act; a.y_f32 = y_f32_dev; a.ldy = ldy; a.y_bf = (__nv_bfloat16*)y_bf_dev; a.bf_plane = bf_plane; a.ldb = ldb;
  a.planes = planes; a.mix = mix_dev; a.mix_w = mix_w; a.mix_src = mix_src; a.mix_init = mix_init; a.fp16 = fp16;
  cudaError_t e = launch_layernorm(a, (cudaStream_t)stream);
  return e == cudaSuccess ? DZ_OK : fail(DZ_ERR_CUDA, cudaGetErrorString(e));
}

static_assert(sizeof(dz_attn_args) == sizeof(AttnArgs), "dz_attn_args must mirror AttnArgs");

int dz_attention(const dz_attn_args* a, int B, int impl, void* stream) {
  if (!a || B <= 0) return fail(DZ_ERR_INVALID, "bad argument");
  AttnArgs args;
  memcpy(&args, a, sizeof(args));
  cudaError_t e = impl == 0 ? launch_attention_tc(args, B, (cudaStream_t)stream) : launch_attention_simt(args, B, (cudaStream_t)stream);
  return e == cudaSuccess ? DZ_OK : fail(DZ_ERR_CUDA, std::string("attention launch failed: ") + cudaGetErrorString(e) + " " + gemm_last_error());
}

}  // extern "C"
