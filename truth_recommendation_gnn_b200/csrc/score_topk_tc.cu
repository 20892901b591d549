// K5 (tcgen05 form) -- bf16 or e4m3 score contraction + streaming top-k on the tensor cores.
//
// Replaces  scores = torch.mm(user_emb, known_post_emb.T); torch.topk(scores, min(K, n))
// (inference.py:427-428) for batched queries against a large catalogue (BASELINE config 5:
// 4096 x 50M, K = 100).  The [B, P] score matrix is never written: it only ever exists as
// [128 x 128] fp32 accumulator tiles in TMEM.
//
// One persistent CTA (16 warps) per SM; work = (catalogue chunk, 128-query block) items, chunk-major.
//   warp 0      TMA: the item's query block (all k-blocks resident), then catalogue tiles [128 posts x H]
//               through an mbarrier ring (SWIZZLE_128B, K-major)
//   warp 1      one thread issues tcgen05.mma kind::f16 (bf16 in) or kind::f8f6f4 (e4m3 in), fp32
//               accumulate, accumulators double-buffered in TMEM columns [0, 256)
//   warps 4-11  SCAN: lane r of a quarter owns query row r (= TMEM lane r), two warps per quarter take 64
//               columns each: tcgen05.ld, one max tree + one warp vote against the row's K-th best; a lane
//               with a candidate copies its 64 scores into a hand-off slot
//   warps 12-15 HELPER: exact test of the slot against the row's K-th best, candidate queue, bitonic sort +
//               rank merge into the item's sorted list (score desc, id asc), which lives in TMEM columns
//               [256, 512) of the row's own lane -- shared memory stays with the catalogue ring; at the end
//               of an item, rank merge of the item's lists into the rows' GLOBAL lists (the result buffer)
//               under one lock per row
// Tensor-bound: 2*B*P*H flops against 2*P*H bytes of catalogue (AI = B = 4096 flop/B).
// E4M3: one 128-byte k-block holds 128 elements instead of 64 and an MMA covers K = 32 instead of 16, so
// every k-block is issued exactly as in bf16 (4 MMAs, +32 bytes each) over half as many k-blocks: half the
// catalogue bytes and half the tensor time per tile.  Everything after the accumulator is unchanged.
// History and measurements of the earlier forms (v1: selection on the accumulator-reading warps; v2: scan /
// helper split; v4: candidates filtered in registers -- slower at 50M posts, dropped): profiles/README.md.
#include <algorithm>
#include <cfloat>
#include <cstdio>
#include <cstdlib>

#include "tc_common.cuh"

namespace trg {
namespace tc {

constexpr int kQRows = 128;
// TMEM columns: [0,256) two accumulator tiles | [256,384) the row's top-K scores | [384,512) their ids.
// Each query row is one TMEM lane, so a row's sorted list lives in its own lane (K <= 128): the 103 KB
// the lists took in shared memory now hold catalogue ring stages (ablation in profiles/README.md: with
// a 3 x 16 KB ring the TMA + MMA pipeline alone ran at 0.97 us per 128-post tile, 3.4x the MMA time).
constexpr int kTmemColsTopk = 512;
constexpr long long kPadIdTc = 0x7fffffffffffffffLL;

struct ScoreTcParams {
  CUtensorMap q_map;
  CUtensorMap c_map;
  long long n_query, n_cat, id_offset;
  long long tiles_per_split;
  int k, n_splits, kblocks;   // kblocks = H * bytes per element / 128
  int dbg;                    // ablation switches, TRG_DEBUG builds only (TRG_TOPK_DBG): 1 = no selection, 2 = no tcgen05.ld either, 4 = no MMA
  int* thr_shared;            // [B] ordered-int keys of the best published K-th score per query row
  int* locks;                 // [B] one lock per query row's global list
  float* out_vals;            // [B][k] the rows' global top-K lists (= the result), merged into by every item
  long long* out_ids;         // [B][k]
  // exclusion index (EXCL instantiations only; appended so that the fields above keep their offsets)
  const int* excl_rowptr;     // [R + 1]
  const int* excl_ids;        // [nnz] global post ids, ascending within a row
  const long long* query_rows;   // [B] exclusion row of each query, nullable (= the query's own row)
};

// Ablation / cycle-accounting switches alter results; they exist only in -DTRG_DEBUG builds.
#ifdef TRG_DEBUG
#define TRG_TOPK_DBG(p) ((p).dbg)
#else
#define TRG_TOPK_DBG(p) 0
#endif

// float <-> int key whose signed order equals the float order (for atomicMax on scores of any sign)
__device__ __forceinline__ int float_key(float f) {
  int i = __float_as_int(f);
  return i ^ ((i >> 31) & 0x7fffffff);
}
__device__ __forceinline__ float key_float(int k) { return __int_as_float(k ^ ((k >> 31) & 0x7fffffff)); }

__device__ __forceinline__ uint32_t lds32(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts32(uint32_t a, uint32_t v) {
  asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
// first index in ids[lo, hi) (ascending) whose value is >= v
__device__ __forceinline__ int excl_lower_bound(const int* __restrict__ ids, int lo, int hi, long long v) {
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if ((long long)__ldg(ids + mid) < v) lo = mid + 1; else hi = mid;
  }
  return lo;
}
// a ranks before b under (score desc, id asc)
__device__ __forceinline__ bool ranks_before(float sa, uint32_t ia, float sb, uint32_t ib) {
  return sa > sb || (sa == sb && ia < ib);
}

// Warp-cooperative merge of one row's candidate queue (<= 32 unsorted entries) into that row's
// sorted top-K list (best first, K <= 128): bitonic sort of the candidates across the lanes, then a
// rank merge -- every element's final slot = its own index + the number of elements of the OTHER
// sequence ranking before it (binary searches), so all writes are conflict-free and in place.
// ~200 warp instructions per merge, i.e. a few per candidate, instead of a per-candidate heap walk
// executed by a single lane.  Returns the new list length.
__device__ __forceinline__ int warp_merge_row(uint32_t lv_a, uint32_t li_a, uint32_t qs_a, uint32_t qi_a,
                                              int n_c, int m_l, int K, int lane) {
  float cs = -INFINITY;
  uint32_t ci = 0xffffffffu;
  if (lane < n_c) {
    cs = __uint_as_float(lds32(qs_a + 4u * lane));
    ci = lds32(qi_a + 4u * lane);
  }
#pragma unroll
  for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      const float ps = __shfl_xor_sync(0xffffffffu, cs, j);
      const uint32_t pi = __shfl_xor_sync(0xffffffffu, ci, j);
      const bool up = (lane & k) == 0, lower = (lane & j) == 0;
      const bool mine_first = ranks_before(cs, ci, ps, pi);
      if ((lower == up) != mine_first) { cs = ps; ci = pi; }
    }
  }
  // list entries of this lane: i = lane + 32 t
  float ls[4];
  uint32_t lid[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const int i = lane + 32 * t;
    ls[t] = -INFINITY;
    lid[t] = 0xffffffffu;
    if (i < m_l) {
      ls[t] = __uint_as_float(lds32(lv_a + 4u * i));
      lid[t] = lds32(li_a + 4u * i);
    }
  }
  // candidate (sorted position = lane): number of list entries ranking before it
  int lo = 0, hi = m_l;
  while (lo < hi) {   // warp-uniform trip count bound: log2(128) + 1; lanes may finish early
    const int mid = (lo + hi) >> 1;
    const float s = __uint_as_float(lds32(lv_a + 4u * mid));
    const uint32_t id = lds32(li_a + 4u * mid);
    if (ranks_before(s, id, cs, ci)) lo = mid + 1; else hi = mid;
  }
  const int cpos = lane + lo;
  // list entries: number of (sorted) candidates ranking before each
  int lpos[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    int a = 0, b = n_c;
#pragma unroll
    for (int it = 0; it < 6; ++it) {   // 2^5 = 32 candidates (+1 step to converge)
      const int mid = (a + b) >> 1;
      const float s = __shfl_sync(0xffffffffu, cs, mid & 31);
      const uint32_t id = __shfl_sync(0xffffffffu, ci, mid & 31);
      if (a < b) {
        if (ranks_before(s, id, ls[t], lid[t])) a = mid + 1; else b = mid;
      }
    }
    lpos[t] = lane + 32 * t + a;
  }
  __syncwarp();
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    if (lane + 32 * t < m_l && lpos[t] < K) {
      sts32(lv_a + 4u * lpos[t], __float_as_uint(ls[t]));
      sts32(li_a + 4u * lpos[t], lid[t]);
    }
  }
  if (lane < n_c && cpos < K) {
    sts32(lv_a + 4u * cpos, __float_as_uint(cs));
    sts32(li_a + 4u * cpos, ci);
  }
  __syncwarp();
  return min(K, m_l + n_c);
}

// ---- tile / queue geometry ---------------------------------------------------------------------------
// Tried and measured (config 5, on the v2 form): the query block as a TMEM-resident A operand with 96-post
// tiles so that accumulators (2 x 96), lists (2 x 128) and Q (64 columns) fit the 512 TMEM columns.  Exact, but
// no faster than Q in shared memory at the same tile width (89.6 vs 89.7 ms), and 96-post tiles cost 15 %
// against 128-post ones: the product runs 128-post tiles with Q in shared memory.
constexpr int kTileN2 = 128;                 // posts per accumulator tile
constexpr int kQCap2 = 32;                   // candidates a row queues before they are merged into its list
constexpr uint32_t kListScoreCol2 = 2 * kTileN2, kListIdCol2 = kListScoreCol2 + 128;

// ---- v3: two scan warps per TMEM lane quarter, work-balanced over every SM ---------------------------
// Measured on v2 (profiles/README.md "K5 v2"): per 128-post tile a scan warp spends 430-500 cycles in the
// tcgen05.ld of its 128 columns, 215-260 in the max tree + vote and ~2 400 in every hand-off (12 % of the
// tiles), against ~540 cycles of MMA -- the four scan warps, not the tensor pipe, paced the kernel, and the
// 32 x 4 grid left 20 of the 148 SMs idle.  Here
//   * warps 4-7 (SCAN A) read columns [0, 64) and warps 8-11 (SCAN B) columns [64, 128) of every accumulator
//     tile: half the TMEM read, half the max tree and a 16-store hand-off per warp, on eight warps that sit
//     on all four SM sub-partitions twice -- a scan warp now needs ~half an MMA time per tile, so the
//     accumulator ring (2 tiles) is released early and hand-offs are absorbed by the slack;
//   * warps 12-15 (HELPER) own queues and lists exactly as in v2 (no locks), polling the two hand-off rings
//     of their quarter;
//   * the grid is one CTA per SM; the catalogue is cut into S chunks with S x (query blocks) a multiple of the
//     grid (32 blocks on 148 SMs: S = 37, 8 items per CTA) and a CTA walks its items one after the other (a
//     SEGMENT each: Q reload, fresh lists, its own slot of partial lists) -- every SM busy instead of 128 of
//     148, and all query blocks stream the same chunks at the same time (see next_segment).
constexpr int kHalfN3 = kTileN2 / 2;           // columns per scan warp
constexpr int kSlotRing3 = 8;                  // slots per ring; one ring per scan warp
constexpr int kSlotWords3 = kHalfN3 + 4;       // scores + header (lane, base index, valid columns)

struct Seg3 { long long qb; long long tile0; int n_tiles; int slot; };
// Work items = (catalogue chunk, query block), chunk-major; CTA j takes items j, j + grid, j + 2 grid, ...
// At any time the resident CTAs therefore work on a few CONSECUTIVE chunks, every chunk being streamed by all
// query blocks at once: the catalogue is read from DRAM about once and served to the other query blocks by
// the L2 (a partition in which every CTA streams its own region -- contiguous tile ranges -- re-reads it once
// per query block: 410 GB instead of 12.8 GB at config 5, measured HBM-bound at 86 ms).
__device__ __forceinline__ bool next_segment(const ScoreTcParams& p, long long n_tiles_total, long long n_qb,
                                             long long& item, Seg3& sg) {
  if (item >= (long long)p.n_splits * n_qb) return false;
  const long long chunk = item / n_qb;
  sg.qb = item - chunk * n_qb;
  sg.tile0 = chunk * p.tiles_per_split;
  const long long left = n_tiles_total - sg.tile0;
  sg.n_tiles = (int)(left < p.tiles_per_split ? (left > 0 ? left : 0) : p.tiles_per_split);
  sg.slot = (int)chunk;
  item += gridDim.x;
  return true;
}

// Merge a finished item's list of one query row (m_l entries, best first, in shared memory; ids relative to
// `idbase`) into that row's GLOBAL list -- the kernel's result, [K] scores + [K] int64 ids in global memory --
// under the row's lock.  Both lists are sorted and ids are unique (an item only holds posts of its own chunk),
// so every entry's final slot is its own index plus the number of entries of the other list that rank before
// it (binary searches): a rank merge whose writes never collide.  The new K-th best is published
// (thr_shared), so the items that start later filter with the exact K-th best of everything finished so far.
// Why: with per-item lists that restart empty and only share the K-th best of ONE chunk's list, every item
// inserted >= K candidates per row again (37 chunks x ~150 insertions per row at config 5) and the candidate
// work was a fixed ~21 ms whatever the catalogue size (65.6 ms at 50M posts, 29.9 ms at 10M: r2 same-box A/B);
// with the global K-th best the later items insert K x chunk / seen.  gs / gid: scratch for 128 scores / ids.
// Returns the K-th best score of the merged global list (-inf while it holds fewer than K entries).
__device__ __forceinline__ float merge_into_global(const ScoreTcParams& p, long long gq, uint32_t lv_a, uint32_t li_a,
                                                   long long idbase, float* gs, long long* gid, int m_l, int K,
                                                   int lane) {
  if (lane == 0) {
    while (atomicCAS(p.locks + gq, 0, 1) != 0) __nanosleep(100);
    __threadfence();
  }
  __syncwarp();
  float* gv = p.out_vals + gq * K;
  long long* gi = p.out_ids + gq * K;
  float s_g[4];
  long long id_g[4];
  int mg = 0;
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const int i = lane + 32 * t;
    s_g[t] = -INFINITY;
    id_g[t] = kPadIdTc;
    if (i < K) {
      s_g[t] = __ldcg(gv + i);
      id_g[t] = __ldcg(gi + i);
    }
    mg += __popc(__ballot_sync(0xffffffffu, id_g[t] != kPadIdTc));
    gs[i] = s_g[t];
    gid[i] = id_g[t];
  }
  __syncwarp();
  // global entries: number of local entries ranking before each
  int pos_g[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    int lo = 0, hi = m_l;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      const float s = __uint_as_float(lds32(lv_a + 4u * mid));
      const long long id = idbase + (long long)lds32(li_a + 4u * mid);
      if (s > s_g[t] || (s == s_g[t] && id < id_g[t])) lo = mid + 1; else hi = mid;
    }
    pos_g[t] = lane + 32 * t + lo;
  }
  // local entries: number of global entries ranking before each
  float s_l[4];
  long long id_l[4];
  int pos_l[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const int i = lane + 32 * t;
    s_l[t] = -INFINITY;
    id_l[t] = kPadIdTc;
    pos_l[t] = K;
    if (i < m_l) {
      s_l[t] = __uint_as_float(lds32(lv_a + 4u * i));
      id_l[t] = idbase + (long long)lds32(li_a + 4u * i);
      int lo = 0, hi = mg;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (gs[mid] > s_l[t] || (gs[mid] == s_l[t] && gid[mid] < id_l[t])) lo = mid + 1; else hi = mid;
      }
      pos_l[t] = i + lo;
    }
  }
  __syncwarp();
  int kth_key = (int)0x80000000;          // below every float key
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    if (lane + 32 * t < mg && pos_g[t] < K) {
      gv[pos_g[t]] = s_g[t];
      gi[pos_g[t]] = id_g[t];
      if (pos_g[t] == K - 1) {
        kth_key = float_key(s_g[t]);
        atomicMax(p.thr_shared + gq, kth_key);
      }
    }
    if (pos_l[t] < K) {
      gv[pos_l[t]] = s_l[t];
      gi[pos_l[t]] = id_l[t];
      if (pos_l[t] == K - 1) {
        kth_key = float_key(s_l[t]);
        atomicMax(p.thr_shared + gq, kth_key);
      }
    }
  }
  __threadfence();
  __syncwarp();
  if (lane == 0) atomicExch(p.locks + gq, 0);
  kth_key = __reduce_max_sync(0xffffffffu, kth_key);
  return kth_key == (int)0x80000000 ? -INFINITY : key_float(kth_key);
}

// EXCL: the helper warps' exact test also rejects the posts of each query row's exclusion list, so no
// excluded post ever enters a list -- per-item lists, flushed global lists, row_thr and thr_shared then only
// ever hold admissible posts, and every threshold below stays the exact K-th best of what may be returned.
// The scan warps' filter (max against those thresholds) remains a superset test and is unchanged.
// E4M3: both operands are e4m3 bytes (kind::f8f6f4); otherwise bf16 (kind::f16).
template <int NS, bool EXCL, bool E4M3>
__global__ void __launch_bounds__(512, 1)
    score_topk_tc3_kernel(const __grid_constant__ ScoreTcParams p, int n_stages) {
  constexpr int N = kTileN2;
  constexpr int kElemsPerKb = E4M3 ? 128 : 64;   // elements in one 128-byte k-block
  constexpr int kSub = N / NS;
  constexpr int kChains = 8;
  constexpr int kQStride = kQCap2 + 1;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>(
      (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  const int q_bytes = p.kblocks * kQRows * 128;
  const int stage_bytes = p.kblocks * NS * 128;
  unsigned char* q_smem = smem;
  unsigned char* ring = smem + q_bytes;
  uint32_t* slots = reinterpret_cast<uint32_t*>(ring + (size_t)n_stages * stage_bytes);   // [8 rings][kSlotRing3][kSlotWords3]
  float* sv = reinterpret_cast<float*>(slots + 8 * kSlotRing3 * kSlotWords3);            // merge scratch [4][128]
  uint32_t* si = reinterpret_cast<uint32_t*>(sv + 4 * 128);
  float* cq_s = reinterpret_cast<float*>(si + 4 * 128);                                  // [128][kQStride]
  uint32_t* cq_i = reinterpret_cast<uint32_t*>(cq_s + kQRows * kQStride);
  long long* g_id = reinterpret_cast<long long*>(
      (reinterpret_cast<uintptr_t>(cq_i + kQRows * kQStride) + 7) & ~static_cast<uintptr_t>(7));   // global-list scratch [4][128] ids
  float* g_s = reinterpret_cast<float*>(g_id + 4 * 128);                                 //                     [4][128] scores
  uint2* row_thr = reinterpret_cast<uint2*>(g_s + 4 * 128);                              // (K-th score, K-th id)
  float* row_tg = reinterpret_cast<float*>(row_thr + kQRows);                            // threshold of the other CTAs
  volatile int* ctl = reinterpret_cast<volatile int*>(row_tg + kQRows);                  // [8 rings][4]: head, tail, done
  uint64_t* bars = reinterpret_cast<uint64_t*>(const_cast<int*>(ctl) + 32);
  uint64_t* full = bars;          // [8]
  uint64_t* empty = full + 8;     // [8]
  uint64_t* q_full = empty + 8;   // [1]
  uint64_t* q_free = q_full + 1;  // [1] every MMA of the segment has read Q
  uint64_t* tmem_full = q_free + 1;   // [2]
  uint64_t* tmem_empty = tmem_full + 2;  // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long n_tiles_total = (p.n_cat + N - 1) / N;
  const long long n_qb = (p.n_query + kQRows - 1) / kQRows;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.q_map);
    tma_prefetch_desc(&p.c_map);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < n_stages; ++s) {
      mbar_init(smem_u32(&full[s]), 1);
      mbar_init(smem_u32(&empty[s]), 1);
    }
    mbar_init(smem_u32(q_full), 1);
    mbar_init(smem_u32(q_free), 1);
    for (int a = 0; a < 2; ++a) {
      mbar_init(smem_u32(&tmem_full[a]), 1);
      mbar_init(smem_u32(&tmem_empty[a]), 256);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(smem_u32(tmem_slot), kTmemColsTopk);
  if (threadIdx.x >= 128 && threadIdx.x < 256) {
    const int r = threadIdx.x - 128;
    row_thr[r] = make_uint2(0xff800000u, 0xffffffffu);   // (-inf, max id): "list not full"
    row_tg[r] = -INFINITY;
    if (r < 32) ctl[r] = 0;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0, seg = 0;
      long long item = blockIdx.x;
      Seg3 sg;
      while (next_segment(p, n_tiles_total, n_qb, item, sg)) {
        if (seg > 0) mbar_wait_backoff(smem_u32(q_free), (seg - 1) & 1);    // the previous segment's MMAs are done with Q
        mbar_arrive_expect_tx(smem_u32(q_full), (uint32_t)q_bytes);
        for (int kb = 0; kb < p.kblocks; ++kb)
          tma_load_2d(smem_u32(q_smem + kb * kQRows * 128), &p.q_map, smem_u32(q_full), kb * kElemsPerKb,
                      (int)(sg.qb * kQRows));
        for (int t = 0; t < sg.n_tiles * kSub; ++t) {
          mbar_wait_backoff(smem_u32(&empty[stage]), phase ^ 1);
          const uint32_t fb = smem_u32(&full[stage]);
          mbar_arrive_expect_tx(fb, (uint32_t)stage_bytes);
          const int row = (int)(sg.tile0 * N + (long long)t * NS);
          for (int kb = 0; kb < p.kblocks; ++kb)
            tma_load_2d(smem_u32(ring + (size_t)stage * stage_bytes + kb * NS * 128), &p.c_map, fb, kb * kElemsPerKb,
                        row);
          if (++stage == n_stages) { stage = 0; phase ^= 1; }
        }
        ++seg;
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(E4M3 ? kFmtE4M3 : kFmtBF16, 0, 0, kQRows, NS);
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0, seg = 0;
      long long item = blockIdx.x;
      Seg3 sg;
      while (next_segment(p, n_tiles_total, n_qb, item, sg)) {
        mbar_wait(smem_u32(q_full), seg & 1);
        for (int t = 0; t < sg.n_tiles; ++t) {
          mbar_wait_backoff(smem_u32(&tmem_empty[acc]), acc_phase ^ 1);
          tc_fence_after();
          for (int sub = 0; sub < kSub; ++sub) {
            mbar_wait_backoff(smem_u32(&full[stage]), phase);
            tc_fence_after();
            const uint32_t d = tmem_base + (uint32_t)(acc * N + sub * NS);
            for (int kb = 0; kb < p.kblocks; ++kb) {
              const uint64_t qd = make_smem_desc_sw128(smem_u32(q_smem + kb * kQRows * 128), 0, 1024);
              const uint64_t cd = make_smem_desc_sw128(smem_u32(ring + (size_t)stage * stage_bytes + kb * NS * 128), 0, 1024);
              if (!(TRG_TOPK_DBG(p) & 4)) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  if constexpr (E4M3)
                    umma_ss_f8f6f4(d, qd + (uint64_t)(2 * k), cd + (uint64_t)(2 * k), idesc, (kb | k) ? 1u : 0u);
                  else
                    umma_ss<false>(d, qd + (uint64_t)(2 * k), cd + (uint64_t)(2 * k), idesc, (kb | k) ? 1u : 0u);
                }
              }
            }
            umma_commit(smem_u32(&empty[stage]));
            if (++stage == n_stages) { stage = 0; phase ^= 1; }
          }
          umma_commit(smem_u32(&tmem_full[acc]));
          if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        umma_commit(smem_u32(q_free));
        ++seg;
      }
    }
  } else if (warp >= 4 && warp < 12) {
    // ===================== SCAN: one query row x 64 columns per thread, fast path only =====================
    const int wq = warp & 3;
    const int half = (warp - 4) >> 2;                 // 0: columns [0, 64), 1: [64, 128)
    const int rg = half * 4 + wq;                     // this warp's hand-off ring
    const int r = wq * 32 + lane;
    const uint32_t thr_addr = smem_u32(row_thr + r);
    const uint32_t slot_base = smem_u32(slots + rg * kSlotRing3 * kSlotWords3);
    volatile int* c_head = ctl + rg * 4 + 0;
    volatile int* c_tail = ctl + rg * 4 + 1;
    volatile int* c_done = ctl + rg * 4 + 2;
    int head = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    int seg = 0;
    long long item = blockIdx.x;
    Seg3 sg;
    while (next_segment(p, n_tiles_total, n_qb, item, sg)) {
      const long long q0 = sg.qb * kQRows;
      const bool row_ok = q0 + r < p.n_query;
      float thr_g = row_ok ? -INFINITY : INFINITY;    // rows past B (zero-filled by TMA) never produce candidates
      for (int t = 0; t < sg.n_tiles; ++t) {
        int tg_key = 0;
        const bool refresh = (t & 15) == 0 && row_ok;
        if (refresh) tg_key = __ldcg(p.thr_shared + q0 + r);
        mbar_wait(smem_u32(&tmem_full[acc]), acc_phase);
        tc_fence_after();
        const long long p0 = (sg.tile0 + t) * N + half * kHalfN3;        // first post of this half tile
        const long long left = p.n_cat - p0;
        const int nvalid = left < (long long)kHalfN3 ? (left > 0 ? (int)left : 0) : kHalfN3;
        const uint32_t base_idx = (uint32_t)(p0 - sg.tile0 * N);
        uint32_t v[kHalfN3];
        const uint32_t t_row = tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(acc * N + half * kHalfN3);
        if (TRG_TOPK_DBG(p) & 2) {
#pragma unroll
          for (int j = 0; j < kHalfN3; ++j) v[j] = 0xff800000u;
        } else {
          tmem_ld_32x32(t_row, v);
          tmem_ld_32x32(t_row + 32u, v + 32);
          tmem_ld_wait();
        }
        tc_fence_before();
        mbar_arrive(smem_u32(&tmem_empty[acc]));      // scores are in registers: hand the buffer back
        if (refresh) {
          thr_g = fmaxf(thr_g, key_float(tg_key));
          if (half == 0) row_tg[r] = thr_g;           // the helper filters with it too
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        if (TRG_TOPK_DBG(p) & 1) {
          if (v[0] == 0x12345678u) head = 1;
          continue;
        }
        uint32_t snap_s, snap_i;
        asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(snap_s), "=r"(snap_i) : "r"(thr_addr) : "memory");
        const float thr = __uint_as_float(snap_s);
        float mx[kChains];
#pragma unroll
        for (int c = 0; c < kChains; ++c) mx[c] = __uint_as_float(v[c]);
#pragma unroll
        for (int j = kChains; j < kHalfN3; ++j) mx[j & (kChains - 1)] = fmaxf(mx[j & (kChains - 1)], __uint_as_float(v[j]));
        float mall = mx[0];
#pragma unroll
        for (int c = 1; c < kChains; ++c) mall = fmaxf(mall, mx[c]);
        const bool cand = nvalid > 0 && mall >= thr && mall >= thr_g;
        unsigned rem = __ballot_sync(0xffffffffu, cand);
        // every lane with a candidate hands its 64 scores to the helper; when more lanes have one than the
        // ring has free slots (the first tiles: every list is still empty) they go in rounds
        while (rem) {
          int space = 0;
          if (lane == 0) {
            while ((space = kSlotRing3 - (head - *c_tail)) <= 0) {
            }
          }
          space = __shfl_sync(0xffffffffu, space, 0);
          const bool pending = (rem >> lane) & 1u;
          const int k = __popc(rem & ((1u << lane) - 1u));
          const bool go = pending && k < space;
          if (go) {
            const uint32_t sa = slot_base + (uint32_t)(((head + k) & (kSlotRing3 - 1)) * kSlotWords3 * 4);
#pragma unroll
            for (int i = 0; i < kHalfN3 / 4; ++i)
              sts128(sa + (uint32_t)(i * 16), make_uint4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]));
            sts128(sa + (uint32_t)(kHalfN3 * 4), make_uint4((uint32_t)lane, base_idx, (uint32_t)nvalid, 0u));
          }
          __syncwarp();
          head += min(__popc(rem), space);
          if (lane == 0) {
            __threadfence_block();
            *c_head = head;
          }
          rem = __ballot_sync(0xffffffffu, pending && !go);
        }
      }
      // end of the segment: tell the helper, then wait until it has written this segment's lists and reset
      // the rows (the next segment is another query block)
      __syncwarp();
      ++seg;
      if (lane == 0) {
        __threadfence_block();
        *c_done = seg;
      }
      asm volatile("bar.sync %0, 96;" ::"r"(1 + wq) : "memory");
    }
  } else if (warp >= 12) {
    // ===================== HELPER: candidates -> queues -> lists (TMEM) =====================
    const int wq = warp & 3;
    const int K = p.k;
    const uint32_t qs_base = smem_u32(cq_s), qi_base = smem_u32(cq_i);
    const uint32_t sv_a = smem_u32(sv + wq * 128), si_a = smem_u32(si + wq * 128);
    const uint32_t tl_s = tmem_base + ((uint32_t)(wq * 32) << 16) + kListScoreCol2;
    const uint32_t tl_i = tmem_base + ((uint32_t)(wq * 32) << 16) + kListIdCol2;
    long long q0 = 0;
    long long idbase = 0;   // global id of the current item's first post
    int cnt = 0;     // lane l: entries in the queue of row 32 wq + l
    int m = 0;       // lane l: entries in the list of row 32 wq + l
    int ex_lo = 0, ex_hi = 0;   // EXCL, lane l: the part of row 32 wq + l's exclusion list inside this item's chunk
    uint32_t ex_first = 0;      //              and its first id (relative to idbase)
    // merge the last `n_c` (<= 32) queue entries of row L into its list (TMEM lane L, staged through scratch)
    auto merge_row = [&](int L, int n_c, int q_off) {
      const int row = wq * 32 + L;
      const int m_l = __shfl_sync(0xffffffffu, m, L);
#pragma unroll 1
      for (int c = 0; c * 16 < m_l; ++c) {
        uint32_t rs[16], ri[16];
        tmem_ld_32x16(tl_s + (uint32_t)(c * 16), rs);
        tmem_ld_32x16(tl_i + (uint32_t)(c * 16), ri);
        tmem_ld_wait();
        if (lane == L) {
#pragma unroll
          for (int j = 0; j < 16; j += 4) {
            sts128(sv_a + 4u * (uint32_t)(c * 16 + j), make_uint4(rs[j], rs[j + 1], rs[j + 2], rs[j + 3]));
            sts128(si_a + 4u * (uint32_t)(c * 16 + j), make_uint4(ri[j], ri[j + 1], ri[j + 2], ri[j + 3]));
          }
        }
      }
      __syncwarp();
      const uint32_t qrow = (uint32_t)(row * kQStride + q_off);
      const int nm = warp_merge_row(sv_a, si_a, qs_base + 4u * qrow, qi_base + 4u * qrow, n_c, m_l, K, lane);
      if (nm == K && q0 + row < p.n_query) {
        // FLUSH: a list that has filled up goes straight into the row's global list (from the scratch the merge
        // left it in: no TMEM write-back) and the row restarts empty, filtered by the K-th best of EVERYTHING
        // every CTA has flushed so far.  The CTAs that work on the same query rows at the same time (4.6 per
        // query block at config 5) thereby share one threshold while they are all still cold, instead of each
        // paying the K ln(n / K) insertions of a private list.  The id of the global K-th best may belong to
        // another chunk, so the row's exact test keeps every candidate that TIES with it (id = max): the
        // global merge ranks them exactly.
        const float kth = merge_into_global(p, q0 + row, sv_a, si_a, idbase, g_s + wq * 128, g_id + wq * 128, nm, K, lane);
        if (lane == L) {
          m = 0;
          asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(smem_u32(row_thr + row)), "r"(__float_as_uint(kth)),
                       "r"(0xffffffffu) : "memory");
        }
        __syncwarp();
        return;
      }
#pragma unroll 1
      for (int c = 0; c * 16 < nm; ++c) {
        uint32_t rs[16], ri[16];
        tmem_ld_32x16(tl_s + (uint32_t)(c * 16), rs);
        tmem_ld_32x16(tl_i + (uint32_t)(c * 16), ri);
        tmem_ld_wait();
        if (lane == L) {
#pragma unroll
          for (int j = 0; j < 16; j += 4) {
            const uint4 a4 = lds128(sv_a + 4u * (uint32_t)(c * 16 + j));
            const uint4 b4 = lds128(si_a + 4u * (uint32_t)(c * 16 + j));
            rs[j] = a4.x; rs[j + 1] = a4.y; rs[j + 2] = a4.z; rs[j + 3] = a4.w;
            ri[j] = b4.x; ri[j + 1] = b4.y; ri[j + 2] = b4.z; ri[j + 3] = b4.w;
          }
        }
        tmem_st_32x16(tl_s + (uint32_t)(c * 16), rs);
        tmem_st_32x16(tl_i + (uint32_t)(c * 16), ri);
      }
      tmem_st_wait();
      if (lane == L) {
        m = nm;
        if (nm == K) {
          const uint32_t ts = lds32(sv_a + 4u * (uint32_t)(K - 1));
          const uint32_t ti = lds32(si_a + 4u * (uint32_t)(K - 1));
          asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(smem_u32(row_thr + row)), "r"(ts), "r"(ti) : "memory");
          if (q0 + row < p.n_query) atomicMax(p.thr_shared + q0 + row, float_key(__uint_as_float(ts)));
        }
      }
      __syncwarp();
    };
    auto drain_row = [&](int L) {      // empty row L's queue, 32 candidates at a time
      int c = __shfl_sync(0xffffffffu, cnt, L);
      while (c > 0) {
        const int n_c = min(c, 32);
        merge_row(L, n_c, c - n_c);
        c -= n_c;
      }
      if (lane == L) cnt = 0;
    };
    // one hand-off slot: 64 scores of row `L` -> queue (exact test against the row's K-th best)
    auto take_slot = [&](uint32_t sa) {
      const uint4 hdr = lds128(sa + (uint32_t)(kHalfN3 * 4));
      const int L = (int)hdr.x;
      const uint32_t base_idx = hdr.y;
      const int nvalid = (int)hdr.z;
      const int row = wq * 32 + L;
      const float tg = *reinterpret_cast<volatile float*>(row_tg + row);
      int x_lo = 0, x_hi = 0;
      uint32_t x_first = 0;
      if constexpr (EXCL) {
        x_lo = __shfl_sync(0xffffffffu, ex_lo, L);
        x_hi = __shfl_sync(0xffffffffu, ex_hi, L);
        x_first = __shfl_sync(0xffffffffu, ex_first, L);
      }
#pragma unroll 1
      for (int i = 0; i < kHalfN3 / 32; ++i) {
        // the row's exact K-th best (it may have moved in the previous sub-step's merge)
        uint32_t ts, ti;
        asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(ts), "=r"(ti) : "r"(smem_u32(row_thr + row)) : "memory");
        const float thr = __uint_as_float(ts);
        const int j = i * 32 + lane;
        const float s = __uint_as_float(lds32(sa + (uint32_t)(j * 4)));
        const uint32_t id = base_idx + (uint32_t)j;
        bool pass = j < nvalid && s >= tg && (s > thr || (s == thr && id < ti));
        if constexpr (EXCL) {
          // the chunk's part of the row's exclusion list is usually empty or one entry, whose id is in a
          // register: a search in global memory only past it, and only by lanes that already pass the exact test
          if (pass && x_lo < x_hi) {
            if (id == x_first) {
              pass = false;
            } else if (id > x_first && x_hi - x_lo > 1) {
              const long long gid = idbase + (long long)id;
              const int at = excl_lower_bound(p.excl_ids, x_lo + 1, x_hi, gid);
              pass = !(at < x_hi && (long long)__ldg(p.excl_ids + at) == gid);
            }
          }
        }
        const unsigned pm = __ballot_sync(0xffffffffu, pass);
        if (pm) {
          const int n = __popc(pm);
          int c = __shfl_sync(0xffffffffu, cnt, L);
          if (c + n > kQCap2) {            // make room: merge what is queued (the threshold only gets tighter;
            drain_row(L);                  // survivors of the stale test are re-ranked exactly by the merge)
            c = 0;
          }
          if (pass) {
            const int k = c + __popc(pm & ((1u << lane) - 1u));
            sts32(qs_base + 4u * (uint32_t)(row * kQStride + k), __float_as_uint(s));
            sts32(qi_base + 4u * (uint32_t)(row * kQStride + k), id);
          }
          __syncwarp();
          if (lane == L) cnt = c + n;
        }
      }
      if (__shfl_sync(0xffffffffu, cnt, L) > 16) drain_row(L);
      __syncwarp();
    };
    int tail[2] = {0, 0};
    int seg = 0;
    long long item = blockIdx.x;
    Seg3 sg;
    while (next_segment(p, n_tiles_total, n_qb, item, sg)) {
      q0 = sg.qb * kQRows;
      idbase = p.id_offset + sg.tile0 * N;
      if constexpr (EXCL) {
        const long long gq = q0 + wq * 32 + lane;
        ex_lo = ex_hi = 0;
        if (gq < p.n_query) {
          const long long er = p.query_rows ? p.query_rows[gq] : gq;
          const int b0 = __ldg(p.excl_rowptr + er), b1 = __ldg(p.excl_rowptr + er + 1);
          ex_lo = excl_lower_bound(p.excl_ids, b0, b1, idbase);
          ex_hi = excl_lower_bound(p.excl_ids, ex_lo, b1, idbase + p.tiles_per_split * N);
          if (ex_lo < ex_hi) ex_first = (uint32_t)(__ldg(p.excl_ids + ex_lo) - idbase);
        }
      }
      for (;;) {
        // poll the two rings of this quarter (SCAN A: ring wq, SCAN B: ring 4 + wq)
        int h[2] = {0, 0}, dn[2] = {0, 0};
        if (lane == 0) {
#pragma unroll
          for (int b = 0; b < 2; ++b) {
            volatile int* c = ctl + (b * 4 + wq) * 4;
            h[b] = c[0];
            if (h[b] == tail[b]) {
              dn[b] = c[2] > seg ? 1 : 0;
              if (dn[b]) h[b] = c[0];      // done is published after the last head
            }
          }
        }
#pragma unroll
        for (int b = 0; b < 2; ++b) {
          h[b] = __shfl_sync(0xffffffffu, h[b], 0);
          dn[b] = __shfl_sync(0xffffffffu, dn[b], 0);
        }
        if (h[0] == tail[0] && h[1] == tail[1]) {
          if (dn[0] && dn[1]) break;
          __nanosleep(64);
          continue;
        }
        __threadfence_block();
#pragma unroll
        for (int b = 0; b < 2; ++b) {
          const uint32_t slot_base = smem_u32(slots + (b * 4 + wq) * kSlotRing3 * kSlotWords3);
          volatile int* c_tail = ctl + (b * 4 + wq) * 4 + 1;
          for (; tail[b] != h[b]; ++tail[b]) {
            take_slot(slot_base + (uint32_t)((tail[b] & (kSlotRing3 - 1)) * kSlotWords3 * 4));
            if (lane == 0) {
              __threadfence_block();
              *c_tail = tail[b] + 1;
            }
          }
        }
      }
      // merge what is left in the queues, then every thread writes its own row's list
      {
        unsigned need = __ballot_sync(0xffffffffu, cnt > 0);
        while (need) {
          const int L = __ffs(need) - 1;
          need &= need - 1;
          drain_row(L);
        }
      }
      {
        // the item is done: merge every row's list into the row's global list (the result)
        const int r = wq * 32 + lane;
        for (int L = 0; L < 32; ++L) {
          const int m_l = __shfl_sync(0xffffffffu, m, L);
          const long long gq = q0 + wq * 32 + L;
          if (m_l == 0 || gq >= p.n_query) continue;
#pragma unroll 1
          for (int c = 0; c * 16 < m_l; ++c) {
            uint32_t rs[16], ri[16];
            tmem_ld_32x16(tl_s + (uint32_t)(c * 16), rs);
            tmem_ld_32x16(tl_i + (uint32_t)(c * 16), ri);
            tmem_ld_wait();
            if (lane == L) {
#pragma unroll
              for (int j = 0; j < 16; j += 4) {
                sts128(sv_a + 4u * (uint32_t)(c * 16 + j), make_uint4(rs[j], rs[j + 1], rs[j + 2], rs[j + 3]));
                sts128(si_a + 4u * (uint32_t)(c * 16 + j), make_uint4(ri[j], ri[j + 1], ri[j + 2], ri[j + 3]));
              }
            }
          }
          __syncwarp();
          merge_into_global(p, gq, sv_a, si_a, idbase, g_s + wq * 128, g_id + wq * 128, m_l, K, lane);
        }
        // fresh rows for the next segment (another query block)
        m = 0;
        cnt = 0;
        row_thr[r] = make_uint2(0xff800000u, 0xffffffffu);
        row_tg[r] = -INFINITY;
      }
      ++seg;
      __threadfence_block();
      asm volatile("bar.sync %0, 96;" ::"r"(1 + wq) : "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, kTmemColsTopk);
}

int make_tmap_2d(CUtensorMap* map, const void* base, int dtype, uint64_t rows, uint64_t cols,
                 uint64_t ld_elems, uint32_t box_rows);

bool score_tc_fits(int row_bytes);
// bf16: H in {64, 128, 192, 256}; e4m3: H in {128, 256} (a 64-byte row would need SWIZZLE_64B)
bool score_tc_eligible(int hidden, int dtype, int k) {
  const bool shape = dtype == TRG_BF16     ? hidden % 64 == 0 && hidden >= 64 && hidden <= 256
                     : dtype == TRG_F8E4M3 ? hidden == 128 || hidden == 256
                                           : false;
  const int row_bytes = hidden * (dtype == TRG_BF16 ? 2 : 1);
  return shape && k >= 1 && k <= 128 && score_tc_fits(row_bytes) && get_encode_tiled() != nullptr;
}

constexpr int kSmemLimit = 227 * 1024;
struct ScoreCfg { int ns, stages, smem; };

// Work partition of v3: S catalogue chunks x (query blocks) items, chunk-major, dealt round-robin to one CTA per
// SM.  S is the smallest count that makes the item count a multiple of the grid (every SM equally loaded),
// bounded so that a chunk keeps >= 8 tiles.  Returns the grid; *tiles_per_chunk, *chunks (= partial-list slots
// per query row).
static int score_tc_partition(int64_t n_query, int64_t n_cat, long long* tiles_per_chunk, int* chunks) {
  const int64_t n_tiles = (n_cat + kTileN2 - 1) / kTileN2;
  const int64_t q_blocks = (n_query + kQRows - 1) / kQRows;
  const int64_t sms = grid_sms();
  int64_t g = sms, b = q_blocks;
  while (b) { const int64_t t = g % b; g = b; b = t; }          // gcd(sms, q_blocks)
  int64_t s = sms / g;                                             // q_blocks * s is a multiple of sms
  s = std::min<int64_t>(s, std::max<int64_t>(1, n_tiles / 8));     // at least ~8 tiles per chunk
  const int64_t tpc = (n_tiles + s - 1) / s;
  s = (n_tiles + tpc - 1) / tpc;                                   // drop empty chunks
  *tiles_per_chunk = tpc;
  *chunks = (int)s;
  return (int)std::min<int64_t>(sms, s * q_blocks);
}

// row_bytes = H * bytes per element: one query / catalogue row, a whole number of 128-byte k-blocks
static int fixed_smem3(int row_bytes) {
  return (row_bytes / 128) * kQRows * 128 + 8 * kSlotRing3 * kSlotWords3 * 4 + 4 * 128 * 8 + kQRows * (kQCap2 + 1) * 8 +
         4 * 128 * 12 /*global-list scratch*/ + kQRows * 12 + 128 + 8 + 1024 + 512;
}
// deep ring first (TMA latency x bandwidth), widest stage that allows it
static ScoreCfg pick_cfg3(int row_bytes) {
  const int fixed = fixed_smem3(row_bytes);
  const int force_ns = debug_env_int("TRG_TOPK_NS", 0);      // TRG_DEBUG builds only: stage width A/B
  for (int min_stages : {4, 2})
    for (int ns : {kTileN2, kTileN2 / 2}) {
      if (force_ns && ns != force_ns) continue;
      const int stage = (row_bytes / 128) * ns * 128;
      const int stages = std::min(8, (kSmemLimit - fixed) / stage);
      if (stages >= min_stages) return {ns, stages, fixed + stages * stage};
    }
  return {0, 0, 0};
}
bool score_tc_fits(int row_bytes) { return pick_cfg3(row_bytes).ns > 0; }

size_t score_tc_workspace_bytes(int64_t n_query, int64_t n_cat, int hidden, int k) {
  (void)n_cat; (void)hidden; (void)k;
  return 2 * align_up((size_t)n_query * 4, 256);       // published thresholds + row locks
}

// the rows' global lists start empty; thresholds at -inf; locks free
__global__ void init_lists(float* vals, long long* ids, long long n, int* thr, int* locks, long long n_query) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    vals[i] = -INFINITY;
    ids[i] = kPadIdTc;
    if (i < n_query) {
      thr[i] = (int)0x807fffff;      // key of -inf
      locks[i] = 0;
    }
  }
}

// with exclusions a row may have fewer than K admissible posts: its list keeps pads, reported as id -1
__global__ void pads_to_minus_one(long long* ids, long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    if (ids[i] == kPadIdTc) ids[i] = -1;
}

template <int NS, bool EXCL, bool E4M3>
static int launch_score3(const ScoreTcParams& p, int grid, int smem, int n_stages, cudaStream_t st) {
  static SmemAttrState attr;
  TRG_CUDA(ensure_dyn_smem(score_topk_tc3_kernel<NS, EXCL, E4M3>, smem, attr));
  score_topk_tc3_kernel<NS, EXCL, E4M3><<<grid, 512, smem, st>>>(p, n_stages);
  return TRG_OK;
}

int score_topk_tc(const void* q, const void* cat, int64_t n_query, int64_t n_cat, int hidden, int dtype, int k,
                  int64_t id_offset, const int32_t* excl_rowptr, const int32_t* excl_ids,
                  const int64_t* query_rows, float* vals_out, int64_t* ids_out, void* ws, size_t ws_bytes,
                  cudaStream_t st) {
  const size_t need = score_tc_workspace_bytes(n_query, n_cat, hidden, k);
  if (!ws || ws_bytes < need) {
    set_error("trg_score_topk: workspace %zu < required %zu", ws_bytes, need);
    return TRG_E_WORKSPACE;
  }
  const bool e4m3 = dtype == TRG_F8E4M3;
  const int row_bytes = hidden * (e4m3 ? 1 : 2);
  const ScoreCfg cfg = pick_cfg3(row_bytes);
  if (cfg.ns == 0) {
    set_error("trg_score_topk(%s): hidden=%d k=%d does not fit in shared memory", e4m3 ? "e4m3" : "bf16", hidden, k);
    return TRG_E_UNSUPPORTED;
  }
  ScoreTcParams p{};
  int rc = make_tmap_2d(&p.q_map, q, dtype, (uint64_t)n_query, hidden, hidden, kQRows);
  if (rc) return rc;
  rc = make_tmap_2d(&p.c_map, cat, dtype, (uint64_t)n_cat, hidden, hidden, cfg.ns);
  if (rc) return rc;
  p.n_query = n_query; p.n_cat = n_cat; p.id_offset = id_offset; p.k = k; p.kblocks = row_bytes / 128;
  p.dbg = debug_env_int("TRG_TOPK_DBG", 0);
  const int grid = score_tc_partition(n_query, n_cat, &p.tiles_per_split, &p.n_splits);
  p.thr_shared = reinterpret_cast<int*>(ws);
  p.locks = reinterpret_cast<int*>(reinterpret_cast<char*>(ws) + align_up((size_t)n_query * 4, 256));
  p.out_vals = vals_out;
  p.out_ids = reinterpret_cast<long long*>(ids_out);
  p.excl_rowptr = excl_rowptr;
  p.excl_ids = excl_ids;
  p.query_rows = reinterpret_cast<const long long*>(query_rows);
  const bool excl = excl_rowptr != nullptr;
  const long long n_out = std::max<long long>((long long)n_query * k, n_query);
  init_lists<<<(unsigned)std::min<long long>(2048, (n_out + 255) / 256), 256, 0, st>>>(
      p.out_vals, p.out_ids, (long long)n_query * k, p.thr_shared, p.locks, n_query);
  count_launch();
  // the EXCL = false instantiations come first: the compiler then emits them instruction for instruction as
  // the kernel was before exclusions existed (instantiated after the EXCL ones, the NS = 64 form came out
  // with a different register assignment); the e4m3 ones come after every bf16 one for the same reason
  if (!e4m3 && !excl)
    rc = cfg.ns == kTileN2 ? launch_score3<kTileN2, false, false>(p, grid, cfg.smem, cfg.stages, st)
                           : launch_score3<kTileN2 / 2, false, false>(p, grid, cfg.smem, cfg.stages, st);
  else if (!e4m3)
    rc = cfg.ns == kTileN2 ? launch_score3<kTileN2, true, false>(p, grid, cfg.smem, cfg.stages, st)
                           : launch_score3<kTileN2 / 2, true, false>(p, grid, cfg.smem, cfg.stages, st);
  else if (!excl)
    rc = cfg.ns == kTileN2 ? launch_score3<kTileN2, false, true>(p, grid, cfg.smem, cfg.stages, st)
                           : launch_score3<kTileN2 / 2, false, true>(p, grid, cfg.smem, cfg.stages, st);
  else
    rc = cfg.ns == kTileN2 ? launch_score3<kTileN2, true, true>(p, grid, cfg.smem, cfg.stages, st)
                           : launch_score3<kTileN2 / 2, true, true>(p, grid, cfg.smem, cfg.stages, st);
  if (rc) return rc;
  count_launch();
  if (excl) {
    const long long n = (long long)n_query * k;
    pads_to_minus_one<<<(unsigned)std::min<long long>(2048, (n + 255) / 256), 256, 0, st>>>(p.out_ids, n);
    count_launch();
  }
  TRG_LAUNCH_OK();
  return TRG_OK;
}

}  // namespace tc
}  // namespace trg
