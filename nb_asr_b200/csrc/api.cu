// C-ABI glue: error reporting, device queries and the GEMM dispatch (bf16 -> tcgen05, fp32 -> SIMT).
#include <cstdarg>
#include <cstdlib>

#include "common.cuh"
#include "kernels.h"

thread_local char g_nbasr_err[512] = {0};

int nbasr_fail(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_nbasr_err, sizeof(g_nbasr_err), fmt, ap);
  va_end(ap);
  return 1;
}

// ---- environment switches, read once at load time
namespace {
struct EnvState {
  bool flag[NBASR_ENV_COUNT];
  int gemm_bn, gemm_l2pf;
  EnvState() {
    static const char* names[NBASR_ENV_COUNT] = {"NBASR_FORCE_SIMT", "NBASR_NO_PDL", "NBASR_GCONV_NO_PREFETCH", "NBASR_LSTM_SS",
                                                 "NBASR_DEBUG", "NBASR_GEMM_DIRECT_EPI"};
    for (int i = 0; i < NBASR_ENV_COUNT; ++i) {
      const char* v = getenv(names[i]);      // set and non-empty and not "0"
      flag[i] = v != nullptr && v[0] != 0 && !(v[0] == '0' && v[1] == 0);
    }
    const char* bn = getenv("NBASR_GEMM_BN");
    gemm_bn = bn ? atoi(bn) : 0;
    const char* pf = getenv("NBASR_GEMM_L2PF");
    gemm_l2pf = pf ? atoi(pf) : 0;
  }
};
const EnvState g_env;
}  // namespace
bool nbasr_env_flag(int which) { return g_env.flag[which]; }
int nbasr_env_gemm_bn() { return g_env.gemm_bn; }
int nbasr_env_gemm_l2pf() { return g_env.gemm_l2pf; }

extern "C" {

const char* nbasr_last_error(void) { return g_nbasr_err; }
int nbasr_version(void) { return 101; }

int nbasr_sm_count(void) {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) sms = 148;
  }
  return sms;
}

int nbasr_gemm_tn(const nbasr_gemm* p, void* stream) {
  if (p->nb <= 0 || p->nr <= 0 || p->N <= 0) return 0;
  if (p->dtype != NBASR_F32 && !nbasr_env_flag(NBASR_ENV_FORCE_SIMT)) return sm100_gemm_tn_pair(p, as_stream(stream));
  NBASR_REQUIRE(p->dtype != NBASR_F16, "the SIMT GEMM takes fp32 / bf16 operands");
  SimtGemmArgs a{};
  a.a = p->a; a.a_dtype = p->dtype; a.a_ib = p->a_bs; a.a_ir = p->a_rs; a.a_kb = 0; a.a_kr = 1;
  a.nib = p->nb; a.nir = p->nr;
  a.b = p->w; a.b_dtype = p->dtype; a.b_j = p->ldw; a.b_kb = 0; a.b_kr = 1;
  a.nkb = 1; a.nkr = p->K; a.N = p->N;
  a.o_r0 = p->o_r0; a.o_bs = p->o_bs; a.o_rs = p->o_rs;
  a.epi = p->epi;
  return simt_gemm_launch(a, as_stream(stream));
}

int nbasr_gemm_wgrad(const nbasr_wgrad* p, void* stream) {
  if (p->nb <= 0 || p->nr <= 0 || p->N <= 0 || p->M <= 0) return 0;
  NBASR_REQUIRE(p->dtype != NBASR_F16, "weight gradients take bf16 (or fp32) operands: dY is a gradient");
  if (p->dtype == NBASR_BF16 && !nbasr_env_flag(NBASR_ENV_FORCE_SIMT)) return sm100_gemm_wgrad_pair(p, as_stream(stream));
  SimtGemmArgs a{};
  a.a = p->dy; a.a_dtype = p->dtype; a.a_ib = 0; a.a_ir = 1; a.a_kb = p->dy_bs; a.a_kr = p->dy_rs;
  a.nib = 1; a.nir = p->M;
  a.b = p->x; a.b_dtype = p->dtype; a.b_j = 1; a.b_kb = p->x_bs; a.b_kr = p->x_rs;
  a.nkb = p->nb; a.nkr = p->nr; a.N = p->N;
  a.o_r0 = 0; a.o_bs = 0; a.o_rs = 1;
  a.epi.out = p->dw; a.epi.out_dtype = NBASR_F32; a.epi.ld_out = p->ldw; a.epi.accumulate = 1;
  if (p->dbias) {   // column sums of dY over rows (b, r): geometry-free call (pointer pre-offset by the pad rows)
    const int es = p->dtype == NBASR_BF16 ? 2 : 4;
    NBASR_REQUIRE(p->dy_rs == p->M, "SIMT bias gradient needs a dense dY row pitch");
    for (int b = 0; b < p->nb; ++b) {
      const char* base = reinterpret_cast<const char*>(p->dy) + (int64_t)b * p->dy_bs * es - (int64_t)NBASR_PAD_L * p->M * es;
      if (nbasr_colsum(p->dtype, base, 1, p->nr, p->nr, p->M, p->dbias, stream)) return 1;
    }
  }
  return simt_gemm_launch(a, as_stream(stream));
}

}  // extern "C"
