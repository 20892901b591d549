// K3 backward, weight half (tcgen05) -- dW_t = alpha_t * dZ^T @ A_t and db = colsum(dZ).
//
// Replaces the dW / db part of autograd through F.linear in loss.backward() (train_gnn.py:283).
// The contraction runs over the node rows, so both MMA operands are read "MN-major" straight
// from the row-major activation tables (no transposes): a 3-D TMA view (32-element column chunk,
// rows, chunk index) lands [chunk][row][128 B] tiles with SWIZZLE_128B, which is exactly the
// canonical MN-major UMMA layout (LBO = rows * 128 B between chunks, SBO = 1024 B between 8-row
// groups).  Each persistent CTA owns a contiguous range of rows, accumulates all terms' [128 x K_t]
// products (and the bias column sums, as one more product against a tile of ones) in TMEM over its
// whole range, and writes one partial; a fixed-order reduction kernel sums the partials, so the
// result is deterministic.  fp32 runs as 3xTF32.  The dZ^T operand (M = hidden, K = rows) is transposed and
// split by the converter warps straight into TENSOR MEMORY (thread m reads column m of the landed dZ tile,
// forms tf32 hi/lo in registers, tcgen05.st into lane m) and the MMAs take it from there (umma_ts); only the
// A_t operand is split in shared memory.  ncu on the all-shared-memory form: ~212 KB of shared-memory
// traffic per 16 rows (1.9 ms of the 2.5 ms at 5 M rows) against 1.2 ms of HBM time; the TMEM operand
// removes the 12 x 4 KB operand reads and the dZ lo plane.
#include <algorithm>

#include "tc_common.cuh"

namespace trg {
namespace tc {

constexpr int kDwMaxTerms = 4;
constexpr int kOnesBytes = 8192;

struct DwParams {
  CUtensorMap dz_map;
  CUtensorMap a_map[kDwMaxTerms];
  int n_terms;
  int term_n[kDwMaxTerms];    // N (= k_t) of each term, multiple of 16, <= 256
  int term_col[kDwMaxTerms];  // first TMEM column of each term's accumulator
  int bias_col;               // TMEM column of the bias accumulator (one 128-byte chunk wide), or -1
  int total_cols;             // columns written to the partial (terms + bias)
  int a_col0;                 // fp32: first TMEM column of the dZ^T operand ring (32 columns per stage)
  int mblock;                 // which 128-wide block of dZ columns (hidden) this launch handles
  long long n_rows;
  long long rows_per_cta;     // multiple of KR
  float* partial;             // [gridDim.x][128][total_cols]
};

template <bool F32>
struct DwCfg {
  static constexpr int KR = F32 ? 16 : 32;                  // rows per stage
  static constexpr int kElemsPerChunk = F32 ? 32 : 64;      // 128 bytes of columns
  static constexpr int kChunkBytes = KR * 128;              // one column chunk of one stage
  static constexpr int kDzBytes = (128 / kElemsPerChunk) * kChunkBytes;   // 128 dZ columns
  static constexpr int kKSteps = 2;                         // KR / (F32 ? 8 : 16)
  static constexpr int kThreads = 256;
};

__device__ __forceinline__ uint32_t lds32_dw(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ float tf32_rna_dw(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

// MN-major operand descriptor.  bf16: SWIZZLE_128B (8-row groups, SBO = 1024 B).  fp32/tf32: the only
// MN-major layout tcgen05 accepts is SWIZZLE_128B_BASE32B (layout type 1: 32-byte swizzle atoms,
// 4-row groups, SBO = 512 B), which TMA produces with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B.
template <bool F32>
__device__ __forceinline__ uint64_t make_mn_desc(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)(((F32 ? 512u : 1024u) >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(F32 ? 1 : 2) << 61;
  return d;
}

// Shared-memory descriptor without swizzle (used for the all-ones tile: any addressing inside the
// region reads 1.0).
__device__ __forceinline__ uint64_t make_smem_desc_noswizzle(uint32_t smem_addr, uint32_t lbo_bytes,
                                                             uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}

template <bool F32>
__global__ void __launch_bounds__(256, 1) proj_dw_kernel(const __grid_constant__ DwParams p,
                                                         int stage_bytes, int n_stages, int tmem_cols) {
  using C = DwCfg<F32>;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>(
      (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  unsigned char* ones = smem + (size_t)n_stages * stage_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(ones + kOnesBytes);
  uint64_t* full = bars;
  uint64_t* ready = full + 8;
  uint64_t* empty = ready + 8;
  uint64_t* done = empty + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row0 = (long long)blockIdx.x * p.rows_per_cta;
  const long long row1 = min(row0 + p.rows_per_cta, p.n_rows);
  const int n_kblocks = row1 > row0 ? (int)((row1 - row0 + C::KR - 1) / C::KR) : 0;

  // per-stage layout.  bf16: dZ | A_0 | A_1 ...   fp32: dZ (raw, linear: it goes to TMEM) | A_0 hi | A_0 lo | ...
  const int plane = F32 ? 2 : 1;
  int term_off[kDwMaxTerms];
  int raw_bytes = C::kDzBytes;
  {
    int off = C::kDzBytes;
    for (int t = 0; t < p.n_terms; ++t) {
      term_off[t] = off;
      const int tb = (p.term_n[t] / C::kElemsPerChunk) * C::kChunkBytes;
      off += plane * tb;
      raw_bytes += tb;
    }
  }

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.dz_map);
    for (int t = 0; t < p.n_terms; ++t) tma_prefetch_desc(&p.a_map[t]);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < n_stages; ++s) {
      mbar_init(smem_u32(&full[s]), 1);
      mbar_init(smem_u32(&ready[s]), 128);
      mbar_init(smem_u32(&empty[s]), 1);
    }
    mbar_init(smem_u32(done), 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(smem_u32(tmem_slot), (uint32_t)tmem_cols);
  {  // tile of ones for the bias column sums (fp32 1.0f or bf16 1.0 pairs), written by every thread
    const uint32_t one = F32 ? 0x3f800000u : 0x3f803f80u;
    for (int i = threadIdx.x; i < kOnesBytes / 4; i += 256) reinterpret_cast<uint32_t*>(ones)[i] = one;
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = 0; kb < n_kblocks; ++kb) {
        mbar_wait_backoff(smem_u32(&empty[stage]), phase ^ 1);
        const uint32_t fb = smem_u32(&full[stage]);
        unsigned char* sb = smem + (size_t)stage * stage_bytes;
        const int r = (int)(row0 + (long long)kb * C::KR);
        mbar_arrive_expect_tx(fb, (uint32_t)raw_bytes);
        tma_load_3d(smem_u32(sb), &p.dz_map, fb, 0, r, p.mblock * (128 / C::kElemsPerChunk));
        for (int t = 0; t < p.n_terms; ++t)
          tma_load_3d(smem_u32(sb + term_off[t]), &p.a_map[t], fb, 0, r, 0);
        if (++stage == n_stages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t lbo = C::kChunkBytes;   // between 128-byte column chunks
      for (int kb = 0; kb < n_kblocks; ++kb) {
        mbar_wait_backoff(smem_u32(F32 ? &ready[stage] : &full[stage]), phase);
        tc_fence_after();
        unsigned char* sb = smem + (size_t)stage * stage_bytes;
        const uint32_t dz_hi = smem_u32(sb);
#pragma unroll
        for (int ks = 0; ks < C::kKSteps; ++ks) {
          const uint32_t koff = (uint32_t)ks * (F32 ? 1024u : 2048u);  // 8 (tf32) / 16 (bf16) rows
          const uint32_t accum = (kb | ks) ? 1u : 0u;
          const uint64_t a_hi = make_mn_desc<F32>(dz_hi + koff, lbo);                     // bf16 only
          const uint32_t ta_hi = tmem_base + (uint32_t)(p.a_col0 + stage * 32 + ks * 8);  // fp32: dZ^T in TMEM
          const uint32_t ta_lo = ta_hi + 16u;
          for (int t = 0; t < p.n_terms; ++t) {
            const uint32_t idesc = make_idesc(F32 ? kFmtTF32 : kFmtBF16, F32 ? 0 : 1, 1, 128, p.term_n[t]);
            const uint32_t tb = (uint32_t)(p.term_n[t] / C::kElemsPerChunk) * C::kChunkBytes;
            const uint32_t b_hi_addr = smem_u32(sb + term_off[t]);
            const uint64_t b_hi = make_mn_desc<F32>(b_hi_addr + koff, lbo);
            const uint32_t d = tmem_base + (uint32_t)p.term_col[t];
            if (F32) {
              const uint64_t b_lo = make_mn_desc<F32>(b_hi_addr + tb + koff, lbo);
              umma_ts<true>(d, ta_lo, b_hi, idesc, accum);
              umma_ts<true>(d, ta_hi, b_lo, idesc, 1u);
              umma_ts<true>(d, ta_hi, b_hi, idesc, 1u);
            } else {
              umma_ss<false>(d, a_hi, b_hi, idesc, accum);
            }
          }
          if (!F32 && p.bias_col >= 0) {     // fp32: the converter warps sum the columns they read anyway
            // column sums of dZ: B = a constant tile of ones, N = 16, addressed exactly like a term
            // with N = one full 128-byte chunk (MN-major, same swizzle mode; every byte of the region is 1.0)
            const uint32_t idesc = make_idesc(F32 ? kFmtTF32 : kFmtBF16, F32 ? 0 : 1, 1, 128, C::kElemsPerChunk);
            // consecutive MMAs get DIFFERENT B start addresses inside the ones region: with an identical
            // B descriptor on back-to-back MMAs every other product came out with a stale B tile
            const uint64_t b1 = make_mn_desc<F32>(smem_u32(ones) + (uint32_t)ks * 4096u, 2048);
            const uint64_t b2 = make_mn_desc<F32>(smem_u32(ones) + (uint32_t)ks * 4096u + 2048u, 2048);
            const uint32_t d = tmem_base + (uint32_t)p.bias_col;
            if (F32) {
              umma_ts<true>(d, ta_lo, b1, idesc, accum);
              umma_ts<true>(d, ta_hi, b2, idesc, 1u);
            } else {
              umma_ss<false>(d, a_hi, b1, idesc, accum);
            }
          }
        }
        umma_commit(smem_u32(&empty[stage]));
        if (++stage == n_stages) { stage = 0; phase ^= 1; }
      }
      umma_commit(smem_u32(done));
    }
  } else if (warp >= 4) {
    const int tid = threadIdx.x - 128;
    float bsum = 0.f;     // fp32: column sum of dZ[:, tid] over this CTA's rows (the bias gradient partial)
    if (F32) {
      // ===================== tf32 converter: dZ^T -> TMEM, A_t hi/lo planes in place =====================
      // The stage's TMEM columns were released together with its shared memory (the MMA's commit on
      // empty[stage] precedes the TMA that filled this stage), so they can be written right away.
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t dz_col = (uint32_t)(tid >> 5) * (uint32_t)C::kChunkBytes + (uint32_t)(tid & 31) * 4u;  // column tid
      for (int kb = 0; kb < n_kblocks; ++kb) {
        mbar_wait(smem_u32(&full[stage]), phase);
        unsigned char* sb = smem + (size_t)stage * stage_bytes;
        {
          uint32_t hi[16], lo[16];
          const uint32_t base = smem_u32(sb) + dz_col;
#pragma unroll
          for (int r = 0; r < 16; ++r) {
            const uint32_t x = lds32_dw(base + (uint32_t)r * 128u);   // dZ[row r][column tid]: a warp reads 128 contiguous bytes
            hi[r] = x & 0xffffe000u;
            lo[r] = __float_as_uint(__uint_as_float(x) - __uint_as_float(hi[r]));
            bsum += __uint_as_float(x);
          }
          tc_fence_after();
          const uint32_t ta = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(p.a_col0 + stage * 32);
          tmem_st_32x16(ta, hi);
          tmem_st_32x16(ta + 16u, lo);
        }
        for (int t = 0; t < p.n_terms; ++t) {
          const int bytes = (p.term_n[t] / C::kElemsPerChunk) * C::kChunkBytes;
          const uint32_t hi = smem_u32(sb + term_off[t]), lo = hi + (uint32_t)bytes;
          for (int i = tid; i < bytes / 16; i += 128) split_tf32_16B(hi + (uint32_t)i * 16u, lo + (uint32_t)i * 16u);
        }
        fence_proxy_async_smem();
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(smem_u32(&ready[stage]));
        if (++stage == n_stages) { stage = 0; phase ^= 1; }
      }
    }
    // ===================== epilogue: TMEM -> this CTA's partial =====================
    const int wq = warp & 3;
    float* out = p.partial + ((size_t)blockIdx.x * 128 + wq * 32 + lane) * p.total_cols;
    if (n_kblocks > 0) {
      mbar_wait(smem_u32(done), 0);
      tc_fence_after();
      for (int c = 0; c < p.total_cols; c += 32) {
        uint32_t r[32];
        tmem_ld_32x32(tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)c, r);
        tmem_ld_wait();
        const int nv = min(32, p.total_cols - c);
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          if (j < nv)
            *reinterpret_cast<float4*>(out + c + j) =
                make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]), __uint_as_float(r[j + 2]),
                            __uint_as_float(r[j + 3]));
      }
      if (F32 && p.bias_col >= 0) out[p.bias_col] = bsum;   // row wq*32+lane of the partial == column tid of dZ
    } else {
      for (int c = 0; c < p.total_cols; c += 4) *reinterpret_cast<float4*>(out + c) = make_float4(0, 0, 0, 0);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, (uint32_t)tmem_cols);
}

// Fixed-order reduction of the per-CTA partials; writes dW_t (dtype) and db (fp32 accumulate).
struct DwReduceArgs {
  const float* partial;
  int n_parts, total_cols, n_terms, bias_col, mblock, f32, hidden;
  int term_n[kDwMaxTerms], term_col[kDwMaxTerms];
  float alpha[kDwMaxTerms];
  void* dw[kDwMaxTerms];   // [hidden, term_n]
  float* db;               // [hidden] fp32 (nullable)
};
__global__ void proj_dw_reduce(const DwReduceArgs a) {
  const int n = 128 * a.total_cols;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int m = i / a.total_cols, c = i % a.total_cols;
    float s = 0.f;
    for (int q = 0; q < a.n_parts; ++q) s += a.partial[(size_t)q * n + i];
    const int h = a.mblock * 128 + m;
    if (h >= a.hidden) continue;   // rows beyond hidden were zero-filled by TMA
    if (a.bias_col >= 0 && c >= a.bias_col) {
      if (c == a.bias_col && a.db) a.db[h] = s;
      continue;
    }
    int t = 0;
    while (t + 1 < a.n_terms && c >= a.term_col[t + 1]) ++t;
    const int f = c - a.term_col[t];
    const float v = s * a.alpha[t];
    if (a.f32)
      reinterpret_cast<float*>(a.dw[t])[(size_t)h * a.term_n[t] + f] = v;
    else
      reinterpret_cast<__nv_bfloat16*>(a.dw[t])[(size_t)h * a.term_n[t] + f] = __float2bfloat16_rn(v);
  }
}

int make_tmap_mn_sw(CUtensorMap* map, const void* base, int dtype, uint64_t rows, uint64_t cols,
                    uint64_t ld_elems, uint32_t box_rows, uint32_t box_chunks, bool swizzle);
int make_tmap_mn(CUtensorMap* map, const void* base, int dtype, uint64_t rows, uint64_t cols,
                 uint64_t ld_elems, uint32_t box_rows, uint32_t box_chunks) {
  return make_tmap_mn_sw(map, base, dtype, rows, cols, ld_elems, box_rows, box_chunks, true);
}
// swizzle = false: the [chunk][row][128 B] tile lands linearly (read by threads, not by the tensor core)
int make_tmap_mn_sw(CUtensorMap* map, const void* base, int dtype, uint64_t rows, uint64_t cols,
                    uint64_t ld_elems, uint32_t box_rows, uint32_t box_chunks, bool swizzle) {
  EncodeTiledFn enc = get_encode_tiled();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled entry point not available");
    return TRG_E_CUDA;
  }
  const int es = dtype == TRG_BF16 ? 2 : 4;
  const uint64_t epc = 128 / es;  // elements per 128-byte chunk
  cuuint64_t gdim[3] = {epc, rows, cols / epc};
  cuuint64_t gstride[2] = {ld_elems * es, 128};
  cuuint32_t box[3] = {(cuuint32_t)epc, box_rows, box_chunks};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, dtype == TRG_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32,
                   3, const_cast<void*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   !swizzle ? CU_TENSOR_MAP_SWIZZLE_NONE
                            : (dtype == TRG_BF16 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B),
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(3d) failed: CUresult %d (rows=%llu cols=%llu ld=%llu)", (int)r,
              (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld_elems);
    return TRG_E_CUDA;
  }
  return TRG_OK;
}

size_t proj_dw_workspace_bytes() { return (size_t)kNumSMs * 128 * 512 * sizeof(float); }

bool proj_dw_eligible(const int* ks, int n_terms, int hidden, int dtype) {
  const int epc = dtype == TRG_BF16 ? 64 : 32;
  if (n_terms < 0 || n_terms > kDwMaxTerms || hidden % epc != 0) return false;
  for (int i = 0; i < n_terms; ++i)
    if (ks[i] <= 0 || ks[i] % epc != 0 || ks[i] > 256) return false;
  return get_encode_tiled() != nullptr;
}

template <bool F32>
int launch_dw(const DwParams& p, int grid, cudaStream_t st) {
  using C = DwCfg<F32>;
  const int plane = F32 ? 2 : 1;
  int stage_bytes = C::kDzBytes;      // fp32: raw dZ only (its hi/lo go to TMEM)
  for (int t = 0; t < p.n_terms; ++t)
    stage_bytes += plane * (p.term_n[t] / C::kElemsPerChunk) * C::kChunkBytes;
  int n_stages = (int)((220 * 1024 - kOnesBytes) / stage_bytes);
  n_stages = std::min(n_stages, 8);
  if (F32) n_stages = std::min(n_stages, (512 - p.a_col0) / 32);   // one 32-column dZ^T slot per stage
  if (n_stages < 2) {
    set_error("proj_dw: stage of %d bytes does not fit twice in shared memory / tensor memory", stage_bytes);
    return TRG_E_UNSUPPORTED;
  }
  int need_cols = F32 ? 512 : p.total_cols, tmem_cols = 32;
  while (tmem_cols < need_cols) tmem_cols <<= 1;
  const int smem = n_stages * stage_bytes + kOnesBytes + 1024 + 256;
  static SmemAttrState attr;
  TRG_CUDA(ensure_dyn_smem(proj_dw_kernel<F32>, smem, attr));
  proj_dw_kernel<F32><<<grid, 256, smem, st>>>(p, stage_bytes, n_stages, tmem_cols);
  count_launch();
  TRG_LAUNCH_OK();
  return TRG_OK;
}

// dW_t = alpha_t * dZ^T A_t  (t < n_terms), db = colsum(dZ) (nullable)
int proj_tc_bwd_weight(const void* dz, const trg_proj_dw_term* terms, int n_terms, float* db,
                       int64_t n_rows, int hidden, int dtype, void* ws, size_t ws_bytes,
                       cudaStream_t st) {
  const bool f32 = dtype == TRG_F32;
  if (!ws || ws_bytes < proj_dw_workspace_bytes()) {
    set_error("trg_sage_proj_bwd_weight: workspace %zu < required %zu", ws_bytes, proj_dw_workspace_bytes());
    return TRG_E_WORKSPACE;
  }
  const int kr = f32 ? 16 : 32;
  const int epc = f32 ? 32 : 64;
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(grid_sms(), (n_rows + kr - 1) / kr));
  int64_t rows_per_cta = (n_rows + grid - 1) / grid;
  rows_per_cta = (rows_per_cta + kr - 1) / kr * kr;

  CUtensorMap dz_map, a_map[kDwMaxTerms];
  // chunks past hidden: OOB -> 0.  fp32: linear landing layout (the converter warps read it, not the MMA)
  int rc = make_tmap_mn_sw(&dz_map, dz, dtype, (uint64_t)n_rows, hidden, hidden, kr, 128 / epc, !f32);
  if (rc) return rc;
  for (int t = 0; t < n_terms; ++t) {
    rc = make_tmap_mn(&a_map[t], terms[t].a, dtype, (uint64_t)n_rows, terms[t].k, terms[t].k, kr,
                      terms[t].k / epc);
    if (rc) return rc;
  }
  // greedy packing of terms into launches of <= 512 TMEM columns, per 128-wide block of hidden
  for (int mb = 0; mb < (hidden + 127) / 128; ++mb) {
    int t0 = 0;
    bool bias_done = db == nullptr;
    while (t0 < n_terms || !bias_done) {
      DwParams p{};
      DwReduceArgs ra{};
      p.dz_map = dz_map;
      int cols = 0, nt = 0;
      const int col_cap = f32 ? 512 - 128 : 512;   // fp32 keeps 4 x 32 columns for the dZ^T operand ring
      while (t0 + nt < n_terms && nt < kDwMaxTerms && cols + terms[t0 + nt].k <= col_cap) {
        p.a_map[nt] = a_map[t0 + nt];
        p.term_n[nt] = terms[t0 + nt].k;
        p.term_col[nt] = cols;
        ra.term_n[nt] = terms[t0 + nt].k; ra.term_col[nt] = cols; ra.alpha[nt] = terms[t0 + nt].alpha;
        ra.dw[nt] = terms[t0 + nt].d_w;
        cols += terms[t0 + nt].k;
        ++nt;
      }
      p.n_terms = nt;
      p.bias_col = -1;
      if (!bias_done && cols + epc <= 512) {   // bias accumulator: N = one 128-byte chunk of ones
        p.bias_col = cols;
        cols += epc;
        bias_done = true;
      }
      if (nt == 0 && p.bias_col < 0) {
        set_error("proj_dw: a term wider than 512 columns cannot be accumulated");
        return TRG_E_UNSUPPORTED;
      }
      p.total_cols = cols; p.mblock = mb; p.n_rows = n_rows; p.rows_per_cta = rows_per_cta;
      // fp32: the bias partial is summed by the converter warps, its columns exist in the partial only
      p.a_col0 = ((f32 && p.bias_col >= 0 ? p.bias_col : cols) + 31) / 32 * 32;
      p.partial = reinterpret_cast<float*>(ws);
      rc = f32 ? launch_dw<true>(p, grid, st) : launch_dw<false>(p, grid, st);
      if (rc) return rc;
      ra.partial = p.partial; ra.n_parts = grid; ra.total_cols = cols; ra.n_terms = nt;
      ra.bias_col = p.bias_col; ra.mblock = mb; ra.f32 = f32; ra.db = db; ra.hidden = hidden;
      proj_dw_reduce<<<(128 * cols + 255) / 256, 256, 0, st>>>(ra);
      count_launch();
      TRG_LAUNCH_OK();
      t0 += nt;
    }
  }
  return TRG_OK;
}

// ---- shape-generic fallback (strict fp32 FMA): same partial + fixed-order reduction scheme ----
template <typename T>
__global__ void __launch_bounds__(256) dw_simt(const T* __restrict__ dz, const T* __restrict__ a,
                                               long long n_rows, int hidden, int k,
                                               long long rows_per_cta, float* __restrict__ partial) {
  __shared__ float zs[16][64 + 1], as[16][64 + 1];
  const int tiles_k = (k + 63) / 64;
  const int h0 = (blockIdx.y / tiles_k) * 64, k0 = (blockIdx.y % tiles_k) * 64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const long long r0 = (long long)blockIdx.x * rows_per_cta, r1 = min(r0 + rows_per_cta, n_rows);
  float acc[4][4] = {};
  for (long long r = r0; r < r1; r += 16) {
    for (int i = threadIdx.x; i < 16 * 64; i += 256) {
      const int rr = i >> 6, c = i & 63;
      const bool ok = r + rr < r1;
      zs[rr][c] = (ok && h0 + c < hidden) ? (float)dz[(r + rr) * hidden + h0 + c] : 0.f;
      as[rr][c] = (ok && k0 + c < k) ? (float)a[(r + rr) * k + k0 + c] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int rr = 0; rr < 16; ++rr)
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(zs[rr][ty * 4 + i], as[rr][tx * 4 + j], acc[i][j]);
    __syncthreads();
  }
  float* out = partial + (size_t)blockIdx.x * hidden * k;
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) {
      const int h = h0 + ty * 4 + i, c = k0 + tx * 4 + j;
      if (h < hidden && c < k) out[(size_t)h * k + c] = acc[i][j];
    }
}
template <typename T>
__global__ void dw_simt_reduce(const float* __restrict__ partial, int n_parts, int n, float alpha,
                               T* __restrict__ out) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int q = 0; q < n_parts; ++q) s += partial[(size_t)q * n + i];
    out[i] = (T)(s * alpha);
  }
}
template <typename T>
__global__ void __launch_bounds__(256) colsum_simt(const T* __restrict__ dz, long long n_rows, int hidden,
                                                   long long rows_per_cta, float* __restrict__ partial) {
  const long long r0 = (long long)blockIdx.x * rows_per_cta, r1 = min(r0 + rows_per_cta, n_rows);
  for (int h = threadIdx.x; h < hidden; h += 256) {
    float s = 0.f;
    for (long long r = r0; r < r1; ++r) s += (float)dz[r * hidden + h];
    partial[(size_t)blockIdx.x * hidden + h] = s;
  }
}

int proj_simt_bwd_weight(const void* dz, const trg_proj_dw_term* terms, int n_terms, float* db,
                         int64_t n_rows, int hidden, int dtype, void* ws, size_t ws_bytes,
                         cudaStream_t st) {
  // one [hidden, k] partial per CTA: wide terms (k up to 512) take fewer CTAs so that the widest
  // term's partials fit the workspace
  int kmax = 1;
  for (int t = 0; t < n_terms; ++t) kmax = std::max(kmax, terms[t].k);
  const int64_t fit = (int64_t)(ws_bytes / ((size_t)hidden * kmax * sizeof(float)));
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>({(int64_t)grid_sms(), (n_rows + 63) / 64, fit}));
  const int64_t rows_per_cta = (n_rows + grid - 1) / grid;
  float* partial = reinterpret_cast<float*>(ws);
  for (int t = 0; t <= n_terms; ++t) {
    const bool bias = t == n_terms;
    if (bias && !db) break;
    const int k = bias ? 1 : terms[t].k;
    if (!ws || ws_bytes < (size_t)grid * hidden * k * sizeof(float)) {
      set_error("trg_sage_proj_bwd_weight: workspace too small for the generic path");
      return TRG_E_WORKSPACE;
    }
    if (bias) {
      if (dtype == TRG_F32)
        colsum_simt<float><<<grid, 256, 0, st>>>((const float*)dz, n_rows, hidden, rows_per_cta, partial);
      else
        colsum_simt<__nv_bfloat16><<<grid, 256, 0, st>>>((const __nv_bfloat16*)dz, n_rows, hidden, rows_per_cta, partial);
      dw_simt_reduce<float><<<(hidden + 255) / 256, 256, 0, st>>>(partial, grid, hidden, 1.f, db);
    } else {
      dim3 g(grid, ((hidden + 63) / 64) * ((k + 63) / 64));
      const int n = hidden * k;
      if (dtype == TRG_F32) {
        dw_simt<float><<<g, 256, 0, st>>>((const float*)dz, (const float*)terms[t].a, n_rows, hidden, k, rows_per_cta, partial);
        dw_simt_reduce<float><<<(n + 255) / 256, 256, 0, st>>>(partial, grid, n, terms[t].alpha, (float*)terms[t].d_w);
      } else {
        dw_simt<__nv_bfloat16><<<g, 256, 0, st>>>((const __nv_bfloat16*)dz, (const __nv_bfloat16*)terms[t].a, n_rows, hidden, k, rows_per_cta, partial);
        dw_simt_reduce<__nv_bfloat16><<<(n + 255) / 256, 256, 0, st>>>(partial, grid, n, terms[t].alpha, (__nv_bfloat16*)terms[t].d_w);
      }
    }
    count_launch(2);
    TRG_LAUNCH_OK();
  }
  return TRG_OK;
}

}  // namespace tc
}  // namespace trg
