// K5 (fp32 SIMT form) -- score contraction + streaming top-k, never materialising [B, P].
//
// Replaces  scores = torch.mm(user_emb, known_post_emb.T); torch.topk(scores, min(K, n))
// at inference.py:427-428 (also train_gnn.py:335-341, test_gnn.py:224-231).
// Total order: score descending, id ascending (torch.topk's tie order is unspecified).
//
// CTA = 32 queries x one catalogue split.  Per 128-post tile: strict-fp32 FMA GEMM out of
// shared memory (4 queries x 4 posts per thread), then each warp filters its 4 query rows
// against the running K-th best score (threshold) and inserts the few survivors into a sorted
// list kept in shared memory (warp-cooperative ballot/shift insert).  Per-split lists are then
// merged by trg_topk_merge.  This is the exact-fp32 path (reference-scale catalogues, odd
// shapes); the bf16 tcgen05 form for 50M-post catalogues is score_topk_tc.cu.
#include <algorithm>
#include <cfloat>
#include <climits>

#include "common.cuh"

namespace trg {
namespace {

constexpr int kThreads = 256;
constexpr int kBQ = 32;     // queries per CTA
constexpr int kBP = 128;    // posts per tile
constexpr int kMaxK = 128;  // list capacity
constexpr long long kPadId = 0x7fffffffffffffffLL;

// a ranks before b under (score desc, id asc)
__device__ __forceinline__ bool before(float sa, long long ia, float sb, long long ib) {
  return sa > sb || (sa == sb && ia < ib);
}

// Warp-cooperative insert of (s, id) into a list sorted best-first, current length *m <= k.
// All 32 lanes call with the same arguments.  Returns the new threshold entry index validity.
__device__ __forceinline__ void warp_insert(float* lv, long long* li, int& m, int k, float s,
                                            long long id, int lane) {
  // position = number of entries ranking before the candidate
  int pos = 0;
  for (int base = 0; base < m; base += 32) {
    const int i = base + lane;
    const bool b = i < m && before(lv[i], li[i], s, id);
    pos += __popc(__ballot_sync(0xffffffffu, b));
  }
  if (pos >= k) return;
  const int new_m = min(m + 1, k);
  // shift [pos, new_m - 1) right by one: read everything first, then write
  float tv[kMaxK / 32];
  long long ti[kMaxK / 32];
#pragma unroll
  for (int r = 0; r < kMaxK / 32; ++r) {
    const int i = r * 32 + lane;
    if (i >= pos && i < new_m - 1) {
      tv[r] = lv[i];
      ti[r] = li[i];
    }
  }
  __syncwarp();
#pragma unroll
  for (int r = 0; r < kMaxK / 32; ++r) {
    const int i = r * 32 + lane;
    if (i >= pos && i < new_m - 1) {
      lv[i + 1] = tv[r];
      li[i + 1] = ti[r];
    }
  }
  if (lane == 0) {
    lv[pos] = s;
    li[pos] = id;
  }
  m = new_m;
  __syncwarp();
}

struct ScoreArgs {
  const float* q;
  const float* cat;
  float* part_vals;      // [B][n_splits][k]
  long long* part_ids;   // [B][n_splits][k]
  int64_t n_query, n_cat, id_offset;
  int hidden, k, n_splits;
  int64_t tiles_per_split;
  // exclusion index (EXCL instantiation only; appended so that the fields above keep their offsets)
  const int32_t* excl_rowptr;   // [R + 1]
  const int32_t* excl_ids;      // [nnz] global post ids, ascending within a row
  const int64_t* query_rows;    // [B] exclusion row of each query, nullable (= the query's own row)
};

// first index in ids[lo, hi) (ascending) whose value is >= v
__device__ __forceinline__ int excl_lower_bound(const int32_t* __restrict__ ids, int lo, int hi, long long v) {
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if ((long long)__ldg(ids + mid) < v) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// dynamic smem: Qs[kBQ][ld] | Ps[kBP][ld] | lv[kBQ][kMaxK] | li[kBQ][kMaxK]
// EXCL: a post of the query row's exclusion list never passes the filter, so the lists (and thresholds)
// only ever hold admissible posts.  The test runs only on lanes that already pass the threshold.
template <bool EXCL>
__global__ void __launch_bounds__(kThreads) score_topk_f32(const ScoreArgs a) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int H = a.hidden, ld = H + 4;
  float* Qs = reinterpret_cast<float*>(smem);
  float* Ps = Qs + kBQ * ld;
  float* lv = Ps + kBP * ld;
  long long* li = reinterpret_cast<long long*>(lv + kBQ * kMaxK);
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int64_t q0 = (int64_t)blockIdx.x * kBQ;
  const int split = blockIdx.y;
  const int hv = H / 4;

  for (int i = tid; i < kBQ * hv; i += kThreads) {
    const int r = i / hv, c = i % hv;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (q0 + r < a.n_query) v = *reinterpret_cast<const float4*>(a.q + (q0 + r) * H + c * 4);
    *reinterpret_cast<float4*>(Qs + r * ld + c * 4) = v;
  }
  int m[4] = {0, 0, 0, 0};
  float thr[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
  bool full[4] = {false, false, false, false};

  const int64_t tile0 = (int64_t)split * a.tiles_per_split;
  const int64_t n_tiles = ceil_div<int64_t>(a.n_cat, kBP);
  const int64_t tile1 = min(tile0 + a.tiles_per_split, n_tiles);
  // EXCL: the part of each of the warp's 4 rows' exclusion lists inside this split's id range, as a cursor
  // [ex_lo, ex_hi) that follows the tiles (ascending ids) and the id at the cursor, ex_v (LLONG_MAX: none left)
  int ex_lo[4] = {0, 0, 0, 0}, ex_hi[4] = {0, 0, 0, 0};
  long long ex_v[4] = {LLONG_MAX, LLONG_MAX, LLONG_MAX, LLONG_MAX};
  if constexpr (EXCL) {
    int lo = 0, hi = 0;
    const int64_t qi = q0 + 4 * w + lane;
    if (lane < 4 && qi < a.n_query) {
      const int64_t er = a.query_rows ? a.query_rows[qi] : qi;
      const int b0 = __ldg(a.excl_rowptr + er), b1 = __ldg(a.excl_rowptr + er + 1);
      lo = excl_lower_bound(a.excl_ids, b0, b1, a.id_offset + tile0 * kBP);
      hi = excl_lower_bound(a.excl_ids, lo, b1, a.id_offset + tile1 * kBP);
    }
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      ex_lo[x] = __shfl_sync(0xffffffffu, lo, x);
      ex_hi[x] = __shfl_sync(0xffffffffu, hi, x);
      if (ex_lo[x] < ex_hi[x]) ex_v[x] = __ldg(a.excl_ids + ex_lo[x]);
    }
  }
  for (int64_t tile = tile0; tile < tile1; ++tile) {
    const int64_t p0 = tile * kBP;
    if constexpr (EXCL) {
      // move each row's cursor to its first excluded id >= this tile's first post (one load per excluded id)
#pragma unroll
      for (int x = 0; x < 4; ++x)
        while (ex_v[x] < a.id_offset + p0) {
          ++ex_lo[x];
          ex_v[x] = ex_lo[x] < ex_hi[x] ? (long long)__ldg(a.excl_ids + ex_lo[x]) : LLONG_MAX;
        }
    }
    __syncthreads();  // previous tile's Ps fully consumed (also orders the Qs fill)
    for (int i = tid; i < kBP * hv; i += kThreads) {
      const int r = i / hv, c = i % hv;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (p0 + r < a.n_cat) v = *reinterpret_cast<const float4*>(a.cat + (p0 + r) * H + c * 4);
      *reinterpret_cast<float4*>(Ps + r * ld + c * 4) = v;
    }
    __syncthreads();
    // warp w owns queries 4w..4w+3; lane owns posts lane, lane+32, lane+64, lane+96
    float acc[4][4];
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
      for (int y = 0; y < 4; ++y) acc[x][y] = 0.f;
    for (int h = 0; h < H; h += 4) {
      float4 qv[4], pv[4];
#pragma unroll
      for (int x = 0; x < 4; ++x) qv[x] = *reinterpret_cast<const float4*>(Qs + (4 * w + x) * ld + h);
#pragma unroll
      for (int y = 0; y < 4; ++y) pv[y] = *reinterpret_cast<const float4*>(Ps + (lane + 32 * y) * ld + h);
#pragma unroll
      for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) {
          acc[x][y] = fmaf(qv[x].x, pv[y].x, acc[x][y]);
          acc[x][y] = fmaf(qv[x].y, pv[y].y, acc[x][y]);
          acc[x][y] = fmaf(qv[x].z, pv[y].z, acc[x][y]);
          acc[x][y] = fmaf(qv[x].w, pv[y].w, acc[x][y]);
        }
    }
    // streaming select; ids ascend with (y, lane) so earlier candidates win ties
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      float* lvx = lv + (4 * w + x) * kMaxK;
      long long* lix = li + (4 * w + x) * kMaxK;
#pragma unroll
      for (int y = 0; y < 4; ++y) {
        const int64_t pid = p0 + lane + 32 * y;
        const float s = acc[x][y];
        const bool valid = pid < a.n_cat;
        bool pass = valid && (!full[x] || s > thr[x]);
        if constexpr (EXCL) {
          // most tiles hold none of the row's excluded ids (ex_v past the tile): a register test
          const long long gid = a.id_offset + pid;
          if (pass && ex_v[x] < a.id_offset + p0 + kBP) {
            if (gid == ex_v[x]) {
              pass = false;
            } else if (gid > ex_v[x]) {
              const int at = excl_lower_bound(a.excl_ids, ex_lo[x] + 1, ex_hi[x], gid);
              pass = !(at < ex_hi[x] && (long long)__ldg(a.excl_ids + at) == gid);
            }
          }
        }
        // excluded lanes stay out of `cand`: the re-filter below only ever clears bits
        unsigned cand = __ballot_sync(0xffffffffu, pass);
        while (cand) {
          const int l = __ffs(cand) - 1;
          const float cs = __shfl_sync(0xffffffffu, s, l);
          const long long cid = a.id_offset + p0 + l + 32 * y;
          warp_insert(lvx, lix, m[x], a.k, cs, cid, lane);
          if (m[x] == a.k) {
            full[x] = true;
            thr[x] = lvx[a.k - 1];
          }
          cand &= cand - 1;
          // re-filter the remaining candidates against the tightened threshold
          cand &= __ballot_sync(0xffffffffu, valid && (!full[x] || s > thr[x]));
        }
      }
    }
  }
  __syncwarp();
#pragma unroll
  for (int x = 0; x < 4; ++x) {
    const int64_t qi = q0 + 4 * w + x;
    if (qi >= a.n_query) continue;
    const float* lvx = lv + (4 * w + x) * kMaxK;
    const long long* lix = li + (4 * w + x) * kMaxK;
    float* ov = a.part_vals + (qi * a.n_splits + split) * a.k;
    long long* oi = a.part_ids + (qi * a.n_splits + split) * a.k;
    for (int i = lane; i < a.k; i += 32) {
      ov[i] = i < m[x] ? lvx[i] : -INFINITY;
      oi[i] = i < m[x] ? lix[i] : kPadId;
    }
  }
}

// One warp per query row: fold n_lists x k_in candidates into the top k_out.
__global__ void __launch_bounds__(kThreads) topk_merge(const float* __restrict__ vin,
                                                       const long long* __restrict__ iin,
                                                       int64_t n_query, int n_lists, int k_in,
                                                       int k_out, float* __restrict__ vout,
                                                       long long* __restrict__ iout) {
  __shared__ float lv[kThreads / 32][kMaxK];
  __shared__ long long li[kThreads / 32][kMaxK];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t qi = (int64_t)blockIdx.x * (kThreads / 32) + w;
  if (qi >= n_query) return;
  const int64_t n = (int64_t)n_lists * k_in;
  const float* v = vin + qi * n;
  const long long* ids = iin + qi * n;
  int m = 0;
  for (int64_t base = 0; base < n; base += 32) {
    const int64_t i = base + lane;
    const float s = i < n ? v[i] : -INFINITY;
    const long long id = i < n ? ids[i] : kPadId;
    bool c = id != kPadId && (m < k_out || before(s, id, lv[w][k_out - 1], li[w][k_out - 1]));
    unsigned cand = __ballot_sync(0xffffffffu, c);
    while (cand) {
      const int l = __ffs(cand) - 1;
      const float cs = __shfl_sync(0xffffffffu, s, l);
      const long long cid = __shfl_sync(0xffffffffu, id, l);
      warp_insert(lv[w], li[w], m, k_out, cs, cid, lane);
      cand &= cand - 1;
    }
  }
  __syncwarp();
  for (int i = lane; i < k_out; i += 32) {
    vout[qi * k_out + i] = i < m ? lv[w][i] : -INFINITY;
    iout[qi * k_out + i] = i < m ? li[w][i] : -1;
  }
}

size_t score_smem_bytes(int hidden) {
  return (size_t)(kBQ + kBP) * (hidden + 4) * 4 + (size_t)kBQ * kMaxK * (4 + 8);
}

int choose_splits(int64_t n_query, int64_t n_cat, int64_t* tiles_per_split) {
  const int64_t n_tiles = ceil_div<int64_t>(n_cat, kBP);
  const int64_t q_blocks = ceil_div<int64_t>(n_query, kBQ);
  int64_t want = ceil_div<int64_t>(2 * kNumSMs, q_blocks);
  int64_t max_splits = std::max<int64_t>(1, n_tiles / 4);
  int64_t s = std::max<int64_t>(1, std::min<int64_t>(want, max_splits));
  s = std::min<int64_t>(s, 65535);
  *tiles_per_split = ceil_div<int64_t>(n_tiles, s);
  return (int)ceil_div<int64_t>(n_tiles, *tiles_per_split);
}

}  // namespace
namespace tc {
bool score_tc_eligible(int hidden, int dtype, int k);
size_t score_tc_workspace_bytes(int64_t n_query, int64_t n_cat, int hidden, int k);
int score_topk_tc(const void* q, const void* cat, int64_t n_query, int64_t n_cat, int hidden, int dtype, int k,
                  int64_t id_offset, const int32_t* excl_rowptr, const int32_t* excl_ids,
                  const int64_t* query_rows, float* vals_out, int64_t* ids_out, void* ws, size_t ws_bytes,
                  cudaStream_t st);
}  // namespace tc

namespace {
template <bool EXCL>
int launch_f32(const ScoreArgs& a, dim3 grid, size_t smem, cudaStream_t st) {
  static SmemAttrState attr;
  TRG_CUDA(ensure_dyn_smem(score_topk_f32<EXCL>, (int)smem, attr));
  score_topk_f32<EXCL><<<grid, kThreads, smem, st>>>(a);
  return TRG_OK;
}
}  // namespace
}  // namespace trg

using namespace trg;

extern "C" size_t trg_score_topk_workspace_bytes(int64_t n_query, int64_t n_cat, int32_t hidden,
                                                 int32_t k) {
  if (n_query <= 0 || n_cat <= 0 || k <= 0) return 256;
  int64_t tps;
  const int splits = choose_splits(n_query, n_cat, &tps);
  const int64_t kk = std::min<int64_t>(k, n_cat);
  const size_t simt = align_up((size_t)n_query * splits * kk * 4, 256) +
                      align_up((size_t)n_query * splits * kk * 8, 256);
  // dtype is not part of this query: size for whichever kernel (fp32 FMA / bf16 or e4m3 tcgen05) needs more;
  // the tcgen05 workspace depends on n_query only, so every dtype's need is covered
  size_t tcb = 0;
  if (hidden % 64 == 0 && hidden <= 256 && kk <= 128)
    tcb = tc::score_tc_workspace_bytes(n_query, n_cat, hidden, (int)kk);
  return std::max(simt, tcb);
}

extern "C" int trg_topk_merge(const float* vals_in, const int64_t* ids_in, int64_t n_query,
                              int32_t n_lists, int32_t k_in, int32_t k_out, float* vals_out,
                              int64_t* ids_out, void* stream) {
  TRG_CHECK_ARG(n_query >= 0 && n_lists > 0 && k_in > 0 && k_out > 0, "trg_topk_merge: bad sizes");
  TRG_CHECK_ARG(k_out <= kMaxK, "trg_topk_merge: k_out=%d > %d", k_out, kMaxK);
  TRG_CHECK_ARG((int64_t)n_lists * k_in >= k_out, "trg_topk_merge: fewer candidates than k_out");
  if (n_query == 0) return TRG_OK;
  TRG_CHECK_ARG(vals_in && ids_in && vals_out && ids_out, "trg_topk_merge: NULL pointer");
  const int64_t grid = ceil_div<int64_t>(n_query, kThreads / 32);
  topk_merge<<<(unsigned)grid, kThreads, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      vals_in, (const long long*)ids_in, n_query, n_lists, k_in, k_out, vals_out,
      (long long*)ids_out);
  count_launch();
  TRG_LAUNCH_OK();
  return TRG_OK;
}

// trg_score_topk and trg_score_topk_excluding: excl_rowptr == NULL means no exclusions (the shipped kernels)
static int score_topk_impl(const char* fn, const void* q, const void* cat, int64_t n_query, int64_t n_cat,
                           int32_t hidden, int dtype, int32_t k, int64_t id_offset, const int32_t* excl_rowptr,
                           const int32_t* excl_ids, const int64_t* query_rows, float* vals_out, int64_t* ids_out,
                           void* workspace, size_t workspace_bytes, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  TRG_CHECK_ARG(n_query >= 0 && n_cat >= 0 && k > 0, "%s: bad sizes", fn);
  if (n_query == 0 || n_cat == 0) return TRG_OK;
  TRG_CHECK_ARG(q && cat && vals_out && ids_out, "%s: NULL pointer", fn);
  TRG_CHECK_ARG(((uintptr_t)q | (uintptr_t)cat) % 16 == 0, "%s: tables must be 16-byte aligned", fn);
  TRG_CHECK_ARG(!excl_rowptr || excl_ids, "%s: excl_ids must be non-NULL when excl_rowptr is given", fn);
  const int kk = (int)std::min<int64_t>(k, n_cat);
  TRG_CHECK_ARG(kk <= kMaxK, "%s: k=%d > %d is not supported", fn, kk, kMaxK);
  if (dtype == TRG_BF16 || dtype == TRG_F8E4M3) {   // tcgen05 only: there is no FMA form for e4m3
    if (!tc::score_tc_eligible(hidden, dtype, kk)) {
      if (dtype == TRG_BF16)
        set_error("%s(bf16): hidden=%d k=%d unsupported: hidden must be in {64,128,192,256}, k <= 128, and the query block (256*hidden B) + the per-row lists (1 KiB*k) + two catalogue stages must fit in 227 KiB of shared memory", fn, hidden, kk);
      else
        set_error("%s(e4m3): hidden=%d k=%d unsupported: hidden must be 128 or 256 and k <= 128", fn, hidden, kk);
      return TRG_E_UNSUPPORTED;
    }
    return tc::score_topk_tc(q, cat, n_query, n_cat, hidden, dtype, kk, id_offset, excl_rowptr, excl_ids,
                             query_rows, vals_out, ids_out, workspace, workspace_bytes, st);
  }
  if (dtype != TRG_F32) {
    set_error("%s: unknown dtype %d", fn, dtype);
    return TRG_E_ARG;
  }
  TRG_CHECK_ARG(hidden > 0 && hidden % 4 == 0 && hidden <= 256,
                "%s(fp32): hidden=%d must be a multiple of 4 and <= 256", fn, hidden);
  const size_t need = trg_score_topk_workspace_bytes(n_query, n_cat, hidden, k);
  if (workspace == nullptr || workspace_bytes < need) {
    set_error("%s: workspace %zu < required %zu", fn, workspace_bytes, need);
    return TRG_E_WORKSPACE;
  }
  ScoreArgs a{};
  a.q = (const float*)q; a.cat = (const float*)cat;
  a.n_query = n_query; a.n_cat = n_cat; a.id_offset = id_offset; a.hidden = hidden; a.k = kk;
  a.n_splits = choose_splits(n_query, n_cat, &a.tiles_per_split);
  a.part_vals = reinterpret_cast<float*>(workspace);
  a.part_ids = reinterpret_cast<long long*>(reinterpret_cast<char*>(workspace) +
                                            align_up((size_t)n_query * a.n_splits * kk * 4, 256));
  a.excl_rowptr = excl_rowptr; a.excl_ids = excl_ids; a.query_rows = query_rows;
  const size_t smem = score_smem_bytes(hidden);
  dim3 grid((unsigned)ceil_div<int64_t>(n_query, kBQ), (unsigned)a.n_splits);
  const int rc = excl_rowptr ? launch_f32<true>(a, grid, smem, st) : launch_f32<false>(a, grid, smem, st);
  if (rc) return rc;
  count_launch();
  TRG_LAUNCH_OK();
  return trg_topk_merge(a.part_vals, (const int64_t*)a.part_ids, n_query, a.n_splits, kk, kk,
                        vals_out, ids_out, stream);
}

extern "C" int trg_score_topk(const void* q, const void* cat, int64_t n_query, int64_t n_cat,
                              int32_t hidden, int dtype, int32_t k, int64_t id_offset,
                              float* vals_out, int64_t* ids_out, void* workspace,
                              size_t workspace_bytes, void* stream) {
  return score_topk_impl("trg_score_topk", q, cat, n_query, n_cat, hidden, dtype, k, id_offset, nullptr, nullptr,
                         nullptr, vals_out, ids_out, workspace, workspace_bytes, stream);
}

extern "C" int trg_score_topk_excluding(const void* q, const void* cat, int64_t n_query, int64_t n_cat,
                                        int32_t hidden, int dtype, int32_t k, int64_t id_offset,
                                        const int32_t* excl_rowptr, const int32_t* excl_ids,
                                        const int64_t* query_rows, float* vals_out, int64_t* ids_out,
                                        void* workspace, size_t workspace_bytes, void* stream) {
  return score_topk_impl("trg_score_topk_excluding", q, cat, n_query, n_cat, hidden, dtype, k, id_offset,
                         excl_rowptr, excl_ids, query_rows, vals_out, ids_out, workspace, workspace_bytes, stream);
}
