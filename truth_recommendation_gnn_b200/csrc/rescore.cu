// Exact re-ranking of per-query candidate lists: the second stage of the e4m3 top-k.
//
// The e4m3 stage (score_topk_tc.cu) selects a short candidate list per query from an 8-bit copy of the
// catalogue.  Here each candidate is re-scored from the dense fp32 / bf16 table with the fp32 FMA kernel's
// chain (s = fmaf(q[h], T[h], s) for h = 0 .. H-1, score_topk.cu), so an fp32 table gives bit for bit the
// score trg_score_topk gives the same (query, post), and the final top-k is taken from those scores by
// trg_topk_merge (every candidate a list of one).
//
// One CTA per query row: the row is staged in shared memory as fp32 (read by every thread at the same
// address: a broadcast), each thread scores one candidate, reading its table row with 16-byte loads.
#include <algorithm>

#include "common.cuh"

namespace trg {
namespace {

constexpr int kThreads = 128;
constexpr long long kPadId = 0x7fffffffffffffffLL;   // what trg_topk_merge skips

template <typename T>
__device__ __forceinline__ float elem(const T& v);
template <>
__device__ __forceinline__ float elem<float>(const float& v) { return v; }
template <>
__device__ __forceinline__ float elem<__nv_bfloat16>(const __nv_bfloat16& v) { return __bfloat162float(v); }

// vals[b][j], ids[b][j] = (score, global id) of candidate j of query b, or (-inf, kPadId) when the id is -1 or
// outside [id_offset, id_offset + n_table)
template <typename T>
__global__ void __launch_bounds__(kThreads) rescore_candidates(const T* __restrict__ q, const T* __restrict__ table,
                                                               int64_t n_table, int hidden,
                                                               const long long* __restrict__ cand, int n_cand,
                                                               int64_t id_offset, float* __restrict__ vals,
                                                               long long* __restrict__ ids) {
  extern __shared__ float qs[];
  constexpr int kVec = 16 / sizeof(T);
  const int64_t b = blockIdx.x;
  for (int h = threadIdx.x; h < hidden; h += kThreads) qs[h] = elem<T>(q[b * hidden + h]);
  __syncthreads();
  for (int j = threadIdx.x; j < n_cand; j += kThreads) {
    const long long g = cand[b * n_cand + j];
    const long long r = g - id_offset;
    float s = -INFINITY;
    long long id = kPadId;
    if (g >= 0 && r >= 0 && r < n_table) {
      const uint4* row = reinterpret_cast<const uint4*>(table + r * hidden);
      s = 0.f;
      for (int c = 0; c < hidden / kVec; ++c) {
        const uint4 v = __ldg(row + c);
        const T* e = reinterpret_cast<const T*>(&v);
#pragma unroll
        for (int i = 0; i < kVec; ++i) s = fmaf(qs[c * kVec + i], elem<T>(e[i]), s);
      }
      id = g;
    }
    vals[b * n_cand + j] = s;
    ids[b * n_cand + j] = id;
  }
}

}  // namespace
}  // namespace trg

using namespace trg;

extern "C" size_t trg_rescore_topk_workspace_bytes(int64_t n_query, int32_t n_cand) {
  if (n_query <= 0 || n_cand <= 0) return 256;
  return align_up((size_t)n_query * n_cand * 4, 256) + align_up((size_t)n_query * n_cand * 8, 256);
}

extern "C" int trg_topk_merge(const float* vals_in, const int64_t* ids_in, int64_t n_query, int32_t n_lists,
                              int32_t k_in, int32_t k_out, float* vals_out, int64_t* ids_out, void* stream);

extern "C" int trg_rescore_topk(const void* q, const void* table, int64_t n_query, int64_t n_table, int32_t hidden,
                                int dtype, const int64_t* cand_ids, int32_t n_cand, int64_t id_offset, int32_t k,
                                float* vals_out, int64_t* ids_out, void* workspace, size_t workspace_bytes,
                                void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  TRG_CHECK_ARG(n_query >= 0 && n_table >= 0 && n_cand > 0 && k > 0, "trg_rescore_topk: bad sizes");
  TRG_CHECK_ARG(dtype == TRG_F32 || dtype == TRG_BF16, "trg_rescore_topk: dtype %d must be fp32 or bf16", dtype);
  const int es = dtype == TRG_BF16 ? 2 : 4;
  TRG_CHECK_ARG(hidden > 0 && (hidden * es) % 16 == 0 && hidden <= 8192,
                "trg_rescore_topk: hidden=%d must make a row a multiple of 16 bytes and be <= 8192", hidden);
  const int kk = std::min(k, n_cand);
  TRG_CHECK_ARG(kk <= 128, "trg_rescore_topk: k=%d > 128 is not supported", kk);
  if (n_query == 0) return TRG_OK;
  TRG_CHECK_ARG(q && cand_ids && vals_out && ids_out && (table || n_table == 0), "trg_rescore_topk: NULL pointer");
  TRG_CHECK_ARG(((uintptr_t)q | (uintptr_t)table) % 16 == 0, "trg_rescore_topk: tables must be 16-byte aligned");
  const size_t need = trg_rescore_topk_workspace_bytes(n_query, n_cand);
  if (!workspace || workspace_bytes < need) {
    set_error("trg_rescore_topk: workspace %zu < required %zu", workspace_bytes, need);
    return TRG_E_WORKSPACE;
  }
  float* sv = reinterpret_cast<float*>(workspace);
  long long* si = reinterpret_cast<long long*>(reinterpret_cast<char*>(workspace) +
                                               align_up((size_t)n_query * n_cand * 4, 256));
  const size_t smem = (size_t)hidden * 4;
  const long long* cand = reinterpret_cast<const long long*>(cand_ids);
  if (dtype == TRG_F32)
    rescore_candidates<float><<<(unsigned)n_query, kThreads, smem, st>>>(
        (const float*)q, (const float*)table, n_table, hidden, cand, n_cand, id_offset, sv, si);
  else
    rescore_candidates<__nv_bfloat16><<<(unsigned)n_query, kThreads, smem, st>>>(
        (const __nv_bfloat16*)q, (const __nv_bfloat16*)table, n_table, hidden, cand, n_cand, id_offset, sv, si);
  count_launch();
  TRG_LAUNCH_OK();
  return trg_topk_merge(sv, (const int64_t*)si, n_query, n_cand, 1, kk, vals_out, ids_out, stream);
}
