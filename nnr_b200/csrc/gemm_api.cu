// nnr_gemm: argument validation and backend dispatch.
#include "common.cuh"
#include "../../include/nnr_b200.h"
#include <stdlib.h>
#include <string.h>

size_t nnr_gemm_simt_workspace_bytes(const nnr_gemm_args* a);
int nnr_gemm_simt(const nnr_gemm_args* a, void* stream);
int nnr_gemm_tc_supported(const nnr_gemm_args* a);
size_t nnr_gemm_tc_workspace_bytes(const nnr_gemm_args* a);
int nnr_gemm_tc(const nnr_gemm_args* a, void* stream);

extern "C" int nnr_gemm_default_algo(void);
static int default_algo() {
  static int algo = -1;
  if (algo < 0) {
    const char* e = getenv("NNR_GEMM_ALGO");
    if (e && !strcmp(e, "simt")) algo = NNR_GEMM_SIMT_FP32;
    else if (e && !strcmp(e, "tf32x3")) algo = NNR_GEMM_TC_TF32X3;
    else if (e && !strcmp(e, "bf16")) algo = NNR_GEMM_TC_BF16;
    else if (e && !strcmp(e, "bf16x3")) algo = NNR_GEMM_TC_BF16X3;
    else algo = NNR_GEMM_TC_BF16X3;   // measured: 6e-6 of max|C| (tf32x3: 1.1e-5), half the operand bytes, 2x MMA rate
  }
  return algo;
}

static int pick_algo(const nnr_gemm_args* a) {
  int algo = a->algo == NNR_GEMM_AUTO ? default_algo() : a->algo;
  if (algo != NNR_GEMM_SIMT_FP32 && !nnr_gemm_tc_supported(a)) {
    // shapes/layouts the tensor-core kernel does not cover run on the exact fp32 kernel; this
    // is still this library's own CUDA kernel, not a fallback to another backend.
    if (a->algo == NNR_GEMM_AUTO) algo = NNR_GEMM_SIMT_FP32;
  }
  return algo;
}

static int validate(const nnr_gemm_args* a) {
  NNR_REQUIRE(a && (a->A || a->A_planes) && (a->B || a->B_planes) && a->C, NNR_ERR_ARG, "nnr_gemm: null operand");
  NNR_REQUIRE(a->M > 0 && a->N > 0 && a->K > 0, NNR_ERR_ARG, "nnr_gemm: bad shape M=%d N=%d K=%d", a->M, a->N, a->K);
  NNR_REQUIRE(a->epilogue >= NNR_EPI_NONE && a->epilogue <= NNR_EPI_ADD_AUX, NNR_ERR_ARG, "nnr_gemm: bad epilogue %d", a->epilogue);
  NNR_REQUIRE(a->lda >= (a->transA ? a->M : a->K), NNR_ERR_ARG, "nnr_gemm: lda too small");
  NNR_REQUIRE(a->ldb >= (a->transB ? a->K : a->N), NNR_ERR_ARG, "nnr_gemm: ldb too small");
  NNR_REQUIRE(a->ldc >= a->N, NNR_ERR_ARG, "nnr_gemm: ldc too small");
  if (a->epilogue == NNR_EPI_BIAS || a->epilogue == NNR_EPI_BIAS_TANH)
    NNR_REQUIRE(a->bias, NNR_ERR_ARG, "nnr_gemm: epilogue needs bias");
  if (a->epilogue == NNR_EPI_GATE)
    NNR_REQUIRE(a->rowbias && a->rowmap && a->aux, NNR_ERR_ARG, "nnr_gemm: gate epilogue needs rowbias,rowmap,aux");
  if (a->epilogue == NNR_EPI_ADD_AUX) NNR_REQUIRE(a->aux, NNR_ERR_ARG, "nnr_gemm: add_aux epilogue needs aux");
  NNR_REQUIRE(a->p_drop >= 0.f && a->p_drop < 1.f, NNR_ERR_ARG, "nnr_gemm: p_drop=%f", a->p_drop);
  return 0;
}

extern "C" int nnr_gemm_default_algo(void) { return default_algo(); }

extern "C" size_t nnr_gemm_workspace_bytes(const nnr_gemm_args* a) {
  if (!a || a->M <= 0 || a->N <= 0 || a->K <= 0) return 0;
  size_t s = nnr_gemm_simt_workspace_bytes(a);
  nnr_gemm_args b = *a;
  b.algo = pick_algo(a);
  size_t t = (b.algo != NNR_GEMM_SIMT_FP32 && nnr_gemm_tc_supported(a)) ? nnr_gemm_tc_workspace_bytes(&b) : 0;
  return s > t ? s : t;
}

extern "C" int nnr_gemm(const nnr_gemm_args* a, void* stream) {
  int rc = validate(a);
  if (rc) return rc;
  int algo = pick_algo(a);
  if (algo == NNR_GEMM_SIMT_FP32) {
    NNR_REQUIRE(a->A && a->B, NNR_ERR_UNSUPPORTED, "nnr_gemm: an operand given only as planes needs the tensor-core path");
    NNR_REQUIRE(!a->C_planes, NNR_ERR_UNSUPPORTED, "nnr_gemm: C_planes needs the tensor-core path");
    return nnr_gemm_simt(a, stream);
  }
  NNR_REQUIRE(nnr_gemm_tc_supported(a), NNR_ERR_UNSUPPORTED, "nnr_gemm: tensor-core path does not support this shape/layout");
  nnr_gemm_args b = *a;
  b.algo = algo;
  return nnr_gemm_tc(&b, stream);
}
