// Library-level entry points of include/trg_b200.h: error string, launch counter, and the
// dispatcher for the projection kernels.
#include <cstdarg>
#include <cstdlib>

#include "common.cuh"

namespace trg {

static thread_local char g_err[512] = "";
std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int proj_simt_launch(const trg_proj_term* terms, int n_terms, const float* bias,
                     const float* row_scale, int64_t n_rows, int hidden, int dtype, int relu, void* out,
                     cudaStream_t st);
namespace tc {
size_t proj_tc_workspace_bytes(int ktot, int hidden, int dtype);
bool proj_tc_eligible(const int* ks, int n_terms, int hidden, int dtype);
int proj_tc_fwd(const trg_proj_term* terms, int n_terms, const float* bias, int64_t n_rows, int hidden,
                int dtype, int relu, void* out, void* ws, size_t ws_bytes, cudaStream_t st);
int proj_tc_bwd_input(const void* dz, const trg_proj_bwd_term* terms, int n_terms, int64_t n_rows,
                      int hidden, int dtype, void* ws, size_t ws_bytes, cudaStream_t st);
int proj_simt_bwd_input(const void* dz, const trg_proj_bwd_term* terms, int n_terms, int64_t n_rows,
                        int hidden, int dtype, void* ws, size_t ws_bytes, cudaStream_t st);
size_t proj_dw_workspace_bytes();
bool proj_dw_eligible(const int* ks, int n_terms, int hidden, int dtype);
int proj_tc_bwd_weight(const void* dz, const trg_proj_dw_term* terms, int n_terms, float* db,
                       int64_t n_rows, int hidden, int dtype, void* ws, size_t ws_bytes, cudaStream_t st);
int proj_simt_bwd_weight(const void* dz, const trg_proj_dw_term* terms, int n_terms, float* db,
                         int64_t n_rows, int hidden, int dtype, void* ws, size_t ws_bytes, cudaStream_t st);
}  // namespace tc

int grid_sms() {
  static std::atomic<int> cache[kMaxDevices];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return kNumSMs;
  const bool tracked = dev >= 0 && dev < kMaxDevices;
  int v = tracked ? cache[dev].load(std::memory_order_relaxed) : 0;
  if (v <= 0) {
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = kNumSMs;
    v = v < kNumSMs ? v : kNumSMs;
    if (tracked) cache[dev].store(v, std::memory_order_relaxed);
  }
  return v;
}

#ifdef TRG_DEBUG
int debug_env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}
#endif

static bool force_simt() { return debug_env_int("TRG_PROJ_FORCE_SIMT", 0) == 1; }

}  // namespace trg

using namespace trg;

extern "C" int trg_abi_version(void) { return TRG_ABI_VERSION; }
extern "C" const char* trg_last_error(void) { return g_err; }
extern "C" int64_t trg_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

extern "C" size_t trg_sage_proj_workspace_bytes(int32_t k_total, int32_t hidden, int dtype) {
  if (k_total <= 0 || hidden <= 0) return 0;
  return tc::proj_tc_workspace_bytes(k_total, hidden, dtype);
}

extern "C" int trg_sage_proj_fwd(const trg_proj_term* terms, int32_t n_terms, const float* bias,
                                 int64_t n_rows, int32_t hidden, int dtype, int relu, void* out,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  TRG_CHECK_ARG(terms && n_terms >= 1 && n_terms <= 4, "trg_sage_proj_fwd: n_terms=%d not in 1..4", n_terms);
  TRG_CHECK_ARG(dtype == TRG_F32 || dtype == TRG_BF16, "trg_sage_proj_fwd: unknown dtype %d", dtype);
  TRG_CHECK_ARG(n_rows >= 0 && hidden > 0 && hidden % 4 == 0, "trg_sage_proj_fwd: bad n_rows/hidden");
  if (n_rows == 0) return TRG_OK;
  const int es = dtype == TRG_BF16 ? 2 : 4;
  TRG_CHECK_ARG(out && (uintptr_t)out % 16 == 0 && (hidden * es) % 16 == 0,
                "trg_sage_proj_fwd: out must be 16-byte aligned with 16-byte-multiple rows");
  int ks[4];
  for (int i = 0; i < n_terms; ++i) {
    TRG_CHECK_ARG(terms[i].a && terms[i].w && terms[i].k > 0 && (terms[i].k * es) % 16 == 0 &&
                      (uintptr_t)terms[i].a % 16 == 0 && (uintptr_t)terms[i].w % 16 == 0,
                  "trg_sage_proj_fwd: term %d needs 16-byte aligned A/W and 16-byte-multiple rows", i);
    ks[i] = terms[i].k;
  }
  if (!force_simt() && workspace && tc::proj_tc_eligible(ks, n_terms, hidden, dtype))
    return tc::proj_tc_fwd(terms, n_terms, bias, n_rows, hidden, dtype, relu, out, workspace,
                           workspace_bytes, st);
  return proj_simt_launch(terms, n_terms, bias, nullptr, n_rows, hidden, dtype, relu, out, st);
}

extern "C" int trg_sage_proj_bwd_input(const void* dz, const trg_proj_bwd_term* terms, int32_t n_terms,
                                       int64_t n_rows, int32_t hidden, int dtype, void* workspace,
                                       size_t workspace_bytes, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  TRG_CHECK_ARG(terms && n_terms >= 1 && n_terms <= 4, "trg_sage_proj_bwd_input: n_terms=%d not in 1..4", n_terms);
  TRG_CHECK_ARG(dtype == TRG_F32 || dtype == TRG_BF16, "trg_sage_proj_bwd_input: unknown dtype %d", dtype);
  TRG_CHECK_ARG(n_rows >= 0 && hidden > 0, "trg_sage_proj_bwd_input: bad n_rows/hidden");
  if (n_rows == 0) return TRG_OK;
  const int es = dtype == TRG_BF16 ? 2 : 4;
  TRG_CHECK_ARG(dz && (uintptr_t)dz % 16 == 0 && (hidden * es) % 16 == 0,
                "trg_sage_proj_bwd_input: dz must be 16-byte aligned with 16-byte-multiple rows");
  bool same_k = true;
  for (int i = 0; i < n_terms; ++i) {
    TRG_CHECK_ARG(terms[i].w && terms[i].d_a && terms[i].k > 0 && (terms[i].k * es) % 16 == 0 &&
                      (uintptr_t)terms[i].d_a % 16 == 0,
                  "trg_sage_proj_bwd_input: term %d needs 16-byte aligned outputs/rows", i);
    same_k = same_k && terms[i].k == terms[0].k;
  }
  // tensor-core path: A = dz (K = hidden), one n-block of width k per term
  const int kh[1] = {hidden};
  if (!force_simt() && same_k && tc::proj_tc_eligible(kh, 1, terms[0].k, dtype))
    return tc::proj_tc_bwd_input(dz, terms, n_terms, n_rows, hidden, dtype, workspace, workspace_bytes, st);
  return tc::proj_simt_bwd_input(dz, terms, n_terms, n_rows, hidden, dtype, workspace, workspace_bytes, st);
}

extern "C" size_t trg_sage_proj_dw_workspace_bytes(void) { return tc::proj_dw_workspace_bytes(); }

extern "C" int trg_sage_proj_bwd_weight(const void* dz, const trg_proj_dw_term* terms, int32_t n_terms,
                                        float* d_bias, int64_t n_rows, int32_t hidden, int dtype,
                                        void* workspace, size_t workspace_bytes, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  TRG_CHECK_ARG(n_terms >= 0 && n_terms <= 4 && (n_terms == 0 || terms), "trg_sage_proj_bwd_weight: n_terms=%d not in 0..4", n_terms);
  TRG_CHECK_ARG(dtype == TRG_F32 || dtype == TRG_BF16, "trg_sage_proj_bwd_weight: unknown dtype %d", dtype);
  TRG_CHECK_ARG(n_rows >= 0 && hidden > 0 && hidden <= 512, "trg_sage_proj_bwd_weight: bad n_rows/hidden");
  const int es = dtype == TRG_BF16 ? 2 : 4;
  TRG_CHECK_ARG(n_rows == 0 || (dz && (uintptr_t)dz % 16 == 0 && (hidden * es) % 16 == 0),
                "trg_sage_proj_bwd_weight: dz must be 16-byte aligned with 16-byte-multiple rows");
  int ks[4];
  for (int i = 0; i < n_terms; ++i) {
    TRG_CHECK_ARG(terms[i].d_w && terms[i].k > 0 && terms[i].k <= 512 && (n_rows == 0 || terms[i].a),
                  "trg_sage_proj_bwd_weight: bad term %d", i);
    TRG_CHECK_ARG((uintptr_t)terms[i].a % 16 == 0 && (terms[i].k * es) % 16 == 0,
                  "trg_sage_proj_bwd_weight: term %d needs 16-byte aligned rows", i);
    ks[i] = terms[i].k;
  }
  if (n_rows == 0) {   // empty sum over rows: dW = 0, db = 0 (a tensor map cannot have a zero extent)
    for (int i = 0; i < n_terms; ++i)
      TRG_CUDA(cudaMemsetAsync(terms[i].d_w, 0, (size_t)hidden * terms[i].k * es, st));
    if (d_bias) TRG_CUDA(cudaMemsetAsync(d_bias, 0, (size_t)hidden * sizeof(float), st));
    return TRG_OK;
  }
  if (!force_simt() && tc::proj_dw_eligible(ks, n_terms, hidden, dtype))
    return tc::proj_tc_bwd_weight(dz, terms, n_terms, d_bias, n_rows, hidden, dtype, workspace,
                                  workspace_bytes, st);
  return tc::proj_simt_bwd_weight(dz, terms, n_terms, d_bias, n_rows, hidden, dtype, workspace,
                                  workspace_bytes, st);
}
