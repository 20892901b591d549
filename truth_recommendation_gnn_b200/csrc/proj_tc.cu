// K3 (tcgen05 form) -- SAGE projections + relation combine + ReLU on the 5th-gen tensor cores.
//
// Replaces lin_l(mean) + lin_r(x_dst) of each SAGEConv (train_gnn.py:177-184,194-197), the combine
// relu(1.0*direct + 0.75*social) / relu(post_update) (train_gnn.py:187-198) and, run on dZ, the
// input-gradient half of their backward (train_gnn.py:283).
//
//   C_j[rows, BN] = epilogue_j( [A_0 | A_1 | ...][rows, K] @ Bcat[j*BN:(j+1)*BN, K]^T )
//
// One persistent CTA per SM, warp-specialised:
//   warp 0      TMA producer: A tiles [128 rows x 128 B] straight from the activation tables and the
//               matching weight tiles, SWIZZLE_128B, into an mbarrier ring
//   warps 4-7   (fp32 only) split the A tile into tf32 hi / lo planes in shared memory
//   warp 1      one elected thread issues tcgen05.mma: fp32 as 3xTF32 (lo*hi + hi*lo + hi*hi, fp32
//               accurate -- a single kind::tf32 product would miss the 1e-5 tolerance), bf16 as
//               kind::f16; accumulators live in TMEM, double-buffered
//   last 4 warps epilogue: tcgen05.ld -> scale / bias / ReLU -> 128-bit stores
// The tile is tall-skinny (N = hidden <= 256): the kernel is HBM-bound on the activation rows,
// which are read exactly once; weights stay L2-resident.
#include <algorithm>
#include <cstdlib>

#include "tc_common.cuh"

namespace trg {
int proj_simt_launch(const trg_proj_term* terms, int n_terms, const float* bias,
                     const float* row_scale, int64_t n_rows, int hidden, int dtype, int relu, void* out,
                     cudaStream_t st);
namespace tc {

constexpr int BM = 128;
constexpr int kABytes = BM * 128;  // one A tile: 128 rows x 128 bytes
constexpr int kMaxTerms = 4;

struct GemmParams {
  CUtensorMap a_map[kMaxTerms];
  CUtensorMap b_hi_map;
  CUtensorMap b_lo_map;
  int a_kblocks[kMaxTerms];
  int n_a;
  int n_nblk;
  int total_kblocks;
  int relu;
  long long n_rows;
  void* out[kMaxTerms];
  long long ld_out[kMaxTerms];
  const float* row_scale[kMaxTerms];
  const float* bias[kMaxTerms];
};

template <bool F32, int BN>
struct Cfg {
  static constexpr int kBBytes = BN * 128;
  static constexpr int kStageBytes = F32 ? 2 * kABytes + 2 * kBBytes : kABytes + kBBytes;
  static constexpr int kTxBytes = F32 ? kABytes + 2 * kBBytes : kABytes + kBBytes;
  static constexpr int kStagesRaw = (220 * 1024) / kStageBytes;
  static constexpr int kStages = kStagesRaw > 8 ? 8 : kStagesRaw;
  static constexpr int kThreads = F32 ? 384 : 256;
  static constexpr int kEpiWarp0 = F32 ? 8 : 4;
  static constexpr int kTmemCols = 2 * BN < 32 ? 32 : 2 * BN;  // BN in {64,128,256} -> pow2
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align*/ + 256 /*barriers*/;
  static constexpr int kElemsPerKBlock = F32 ? 32 : 64;
};

__device__ __forceinline__ float tf32_rna(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

template <bool F32, int BN>
__global__ void __launch_bounds__(Cfg<F32, BN>::kThreads, 1)
    proj_tc_kernel(const __grid_constant__ GemmParams p) {
  using C = Cfg<F32, BN>;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>(
      (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::kStages * C::kStageBytes);
  uint64_t* full = bars;
  uint64_t* ready = full + C::kStages;
  uint64_t* empty = ready + C::kStages;
  uint64_t* tmem_full = empty + C::kStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long n_tiles = (p.n_rows + BM - 1) / BM;

  if (warp == 0 && lane == 0) {
    for (int t = 0; t < p.n_a; ++t) tma_prefetch_desc(&p.a_map[t]);
    tma_prefetch_desc(&p.b_hi_map);
    if (F32) tma_prefetch_desc(&p.b_lo_map);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < C::kStages; ++s) {
      mbar_init(smem_u32(&full[s]), 1);
      mbar_init(smem_u32(&ready[s]), 128);
      mbar_init(smem_u32(&empty[s]), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(smem_u32(&tmem_full[a]), 1);
      mbar_init(smem_u32(&tmem_empty[a]), 128);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(smem_u32(tmem_slot), C::kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  auto stage_a_hi = [&](int s) { return smem + s * C::kStageBytes; };
  auto stage_a_lo = [&](int s) { return smem + s * C::kStageBytes + kABytes; };
  auto stage_b_hi = [&](int s) { return smem + s * C::kStageBytes + (F32 ? 2 * kABytes : kABytes); };
  auto stage_b_lo = [&](int s) { return smem + s * C::kStageBytes + 2 * kABytes + C::kBBytes; };

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        for (int nb = 0; nb < p.n_nblk; ++nb) {
          int kbt = 0;
          for (int t = 0; t < p.n_a; ++t) {
            for (int kb = 0; kb < p.a_kblocks[t]; ++kb, ++kbt) {
              mbar_wait_backoff(smem_u32(&empty[stage]), phase ^ 1);
              const uint32_t fb = smem_u32(&full[stage]);
              mbar_arrive_expect_tx(fb, C::kTxBytes);
              tma_load_2d(smem_u32(stage_a_hi(stage)), &p.a_map[t], fb, kb * C::kElemsPerKBlock,
                          (int)(tile * BM));
              // the same k-block of this CTA's NEXT tile: start its DRAM fetch into L2 now
              if (nb == p.n_nblk - 1 && tile + gridDim.x < n_tiles)
                tma_prefetch_l2_2d(&p.a_map[t], kb * C::kElemsPerKBlock, (int)((tile + gridDim.x) * BM));
              tma_load_2d(smem_u32(stage_b_hi(stage)), &p.b_hi_map, fb, kbt * C::kElemsPerKBlock,
                          nb * BN);
              if (F32)
                tma_load_2d(smem_u32(stage_b_lo(stage)), &p.b_lo_map, fb, kbt * C::kElemsPerKBlock,
                            nb * BN);
              if (++stage == C::kStages) { stage = 0; phase ^= 1; }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (one thread) =====================
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(F32 ? kFmtTF32 : kFmtBF16, 0, 0, BM, BN);
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0;
      for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        for (int nb = 0; nb < p.n_nblk; ++nb) {
          mbar_wait_backoff(smem_u32(&tmem_empty[acc]), acc_phase ^ 1);
          tc_fence_after();
          const uint32_t d = tmem_base + (uint32_t)(acc * BN);
          for (int kb = 0; kb < p.total_kblocks; ++kb) {
            mbar_wait_backoff(smem_u32(F32 ? &ready[stage] : &full[stage]), phase);
            tc_fence_after();
            const uint64_t a_hi = make_smem_desc_sw128(smem_u32(stage_a_hi(stage)), 0, 1024);
            const uint64_t b_hi = make_smem_desc_sw128(smem_u32(stage_b_hi(stage)), 0, 1024);
            if (F32) {
              const uint64_t a_lo = make_smem_desc_sw128(smem_u32(stage_a_lo(stage)), 0, 1024);
              const uint64_t b_lo = make_smem_desc_sw128(smem_u32(stage_b_lo(stage)), 0, 1024);
#pragma unroll
              for (int k = 0; k < 4; ++k) {  // 4 x (K = 32 bytes) per 128-byte k-block
                const uint64_t o = (uint64_t)(k * 2);  // +32 bytes in the (addr >> 4) field
                umma_ss<true>(d, a_lo + o, b_hi + o, idesc, (kb | k) ? 1u : 0u);
                umma_ss<true>(d, a_hi + o, b_lo + o, idesc, 1u);
                umma_ss<true>(d, a_hi + o, b_hi + o, idesc, 1u);
              }
            } else {
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const uint64_t o = (uint64_t)(k * 2);
                umma_ss<false>(d, a_hi + o, b_hi + o, idesc, (kb | k) ? 1u : 0u);
              }
            }
            umma_commit(smem_u32(&empty[stage]));  // frees the smem slot when these MMAs retire
            if (++stage == C::kStages) { stage = 0; phase ^= 1; }
          }
          umma_commit(smem_u32(&tmem_full[acc]));
          if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
      }
    }
  } else if (F32 && warp >= 4 && warp < 8) {
    // ===================== tf32 hi/lo splitter (128 threads) =====================
    const int tid = threadIdx.x - 128;
    int stage = 0;
    uint32_t phase = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      for (int it = 0; it < p.n_nblk * p.total_kblocks; ++it) {
        mbar_wait(smem_u32(&full[stage]), phase);
        const uint32_t hi = smem_u32(stage_a_hi(stage)) + (uint32_t)tid * 16u;
        const uint32_t lo = smem_u32(stage_a_lo(stage)) + (uint32_t)tid * 16u;
#pragma unroll
        for (int i = 0; i < kABytes / 16 / 128; ++i) split_tf32_16B(hi + i * 2048u, lo + i * 2048u);
        fence_proxy_async_smem();
        mbar_arrive(smem_u32(&ready[stage]));
        if (++stage == C::kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp >= C::kEpiWarp0) {
    // ===================== epilogue (TMEM -> registers -> global) =====================
    const int wq = warp & 3;  // TMEM lane quarter this warp may access
    int acc = 0;
    uint32_t acc_phase = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      for (int nb = 0; nb < p.n_nblk; ++nb) {
        mbar_wait(smem_u32(&tmem_full[acc]), acc_phase);
        tc_fence_after();
        const long long row = tile * BM + wq * 32 + lane;
        const bool in = row < p.n_rows;
        const float rs = (in && p.row_scale[nb]) ? __ldg(p.row_scale[nb] + row) : 1.f;
        const float* bias = p.bias[nb];
#pragma unroll 1
        for (int c = 0; c < BN / 32; ++c) {
          uint32_t r[32];
          tmem_ld_32x32(tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(acc * BN + c * 32), r);
          tmem_ld_wait();
          if (in) {
            float f[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              float v = __uint_as_float(r[j]) * rs;
              if (bias) v += __ldg(bias + c * 32 + j);
              if (p.relu) v = fmaxf(v, 0.f);
              f[j] = v;
            }
            if (F32) {
              float* o = reinterpret_cast<float*>(p.out[nb]) + row * p.ld_out[nb] + c * 32;
#pragma unroll
              for (int j = 0; j < 32; j += 4)
                *reinterpret_cast<float4*>(o + j) = make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]);
            } else {
              __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(p.out[nb]) + row * p.ld_out[nb] + c * 32;
#pragma unroll
              for (int j = 0; j < 32; j += 8)
                *reinterpret_cast<uint4*>(o + j) = Elem<__nv_bfloat16>::pack(f + j);
            }
          }
        }
        tc_fence_before();
        mbar_arrive(smem_u32(&tmem_empty[acc]));
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, C::kTmemCols);
}

// ---- fp32 kernel, v2: the split A operand lives in TENSOR MEMORY -----------------------------------
// ncu on v1 (profiles/README.md, r1_v4): per 128-row tile the shared memory moves ~1.5 MB (TMA writes
// of A + both weight planes, the split's read + two writes, and 12 operand reads of 8 KB per 32-wide
// k-block) against 192 KB of HBM traffic: at 128 B/clk the SM's shared memory, not HBM, set the pace,
// and a 3-stage ring (64 KB per stage) kept too few bytes in flight.  Here the split warps read the
// TMA-landed fp32 tile once (LDS.128, swizzle-aware, conflict-free), form hi/lo in registers and write
// them with tcgen05.st into a 4-stage ring of TMEM columns; the MMAs take A from TMEM (umma_ts) and
// only the weight planes from shared memory.  Shared-memory traffic per tile drops to ~0.9 MB, the A
// landing ring (5 x 16 KB, released by the split warps, not by the MMA) and the weight ring (4 x 32 KB)
// are decoupled, and the epilogue goes through a swizzled staging tile so that every global store
// instruction writes four full 128-byte row segments instead of 32 scattered 16-byte pieces.
template <int BN>
struct CfgA {
  static constexpr int kSA = 5;                       // A landing stages (16 KB each)
  static constexpr int kSB = 4;                       // weight stages (hi + lo planes)
  static constexpr int kST = 4;                       // TMEM A stages (64 columns: hi | lo)
  static constexpr int kBBytes = BN * 128;
  static constexpr int kStageBBytes = 2 * kBBytes;
  static constexpr int kStagingBytes = 4 * 4096;      // one 32-row x 128-byte block per epilogue warp
  static constexpr int kThreads = 384;
  static constexpr int kAccCols = 2 * BN;             // double-buffered accumulator
  static constexpr int kTmemCols = 512;               // accumulators + 4 x 64 A columns (pow2 alloc)
  static constexpr int kSmemBytes = kSA * kABytes + kSB * kStageBBytes + kStagingBytes + 1024 + 256;
  static_assert(kAccCols + kST * 64 <= 512, "TMEM budget");
};

template <int BN>
__global__ void __launch_bounds__(CfgA<BN>::kThreads, 1)
    proj_tc_f32a_kernel(const __grid_constant__ GemmParams p) {
  using C = CfgA<BN>;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>(
      (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  unsigned char* smem_a = smem;
  unsigned char* smem_b = smem_a + C::kSA * kABytes;
  unsigned char* smem_stage = smem_b + C::kSB * C::kStageBBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_stage + C::kStagingBytes);
  uint64_t* a_full = bars;
  uint64_t* a_free = a_full + C::kSA;
  uint64_t* b_full = a_free + C::kSA;
  uint64_t* b_empty = b_full + C::kSB;
  uint64_t* t_full = b_empty + C::kSB;
  uint64_t* t_empty = t_full + C::kST;
  uint64_t* acc_full = t_empty + C::kST;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long n_tiles = (p.n_rows + BM - 1) / BM;

  if (warp == 0 && lane == 0) {
    for (int t = 0; t < p.n_a; ++t) tma_prefetch_desc(&p.a_map[t]);
    tma_prefetch_desc(&p.b_hi_map);
    tma_prefetch_desc(&p.b_lo_map);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < C::kSA; ++s) {
      mbar_init(smem_u32(&a_full[s]), 1);
      mbar_init(smem_u32(&a_free[s]), 128);
    }
    for (int s = 0; s < C::kSB; ++s) {
      mbar_init(smem_u32(&b_full[s]), 1);
      mbar_init(smem_u32(&b_empty[s]), 1);
    }
    for (int s = 0; s < C::kST; ++s) {
      mbar_init(smem_u32(&t_full[s]), 128);
      mbar_init(smem_u32(&t_empty[s]), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(smem_u32(&acc_full[a]), 1);
      mbar_init(smem_u32(&acc_empty[a]), 128);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(smem_u32(tmem_slot), C::kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_a0 = tmem_base + (uint32_t)C::kAccCols;   // first A column

  if (warp == 0) {
    // ===================== TMA producer: activation tiles =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)
        for (int nb = 0; nb < p.n_nblk; ++nb)
          for (int t = 0; t < p.n_a; ++t)
            for (int kb = 0; kb < p.a_kblocks[t]; ++kb) {
              mbar_wait_backoff(smem_u32(&a_free[stage]), phase ^ 1);
              const uint32_t fb = smem_u32(&a_full[stage]);
              mbar_arrive_expect_tx(fb, kABytes);
              tma_load_2d(smem_u32(smem_a + stage * kABytes), &p.a_map[t], fb, kb * 32, (int)(tile * BM));
              if (++stage == C::kSA) { stage = 0; phase ^= 1; }
            }
    }
  } else if (warp == 3) {
    // ===================== TMA producer: weight planes (L2-resident) =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)
        for (int nb = 0; nb < p.n_nblk; ++nb)
          for (int kbt = 0; kbt < p.total_kblocks; ++kbt) {
            mbar_wait_backoff(smem_u32(&b_empty[stage]), phase ^ 1);
            const uint32_t fb = smem_u32(&b_full[stage]);
            mbar_arrive_expect_tx(fb, C::kStageBBytes);
            unsigned char* dst = smem_b + stage * C::kStageBBytes;
            tma_load_2d(smem_u32(dst), &p.b_hi_map, fb, kbt * 32, nb * BN);
            tma_load_2d(smem_u32(dst + C::kBBytes), &p.b_lo_map, fb, kbt * 32, nb * BN);
            if (++stage == C::kSB) { stage = 0; phase ^= 1; }
          }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (one thread) =====================
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(kFmtTF32, 0, 0, BM, BN);
      int sb = 0, st = 0, acc = 0;
      uint32_t pb = 0, pt = 0, acc_phase = 0;
      for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        for (int nb = 0; nb < p.n_nblk; ++nb) {
          mbar_wait_backoff(smem_u32(&acc_empty[acc]), acc_phase ^ 1);
          tc_fence_after();
          const uint32_t d = tmem_base + (uint32_t)(acc * BN);
          for (int kb = 0; kb < p.total_kblocks; ++kb) {
            mbar_wait_backoff(smem_u32(&t_full[st]), pt);
            mbar_wait_backoff(smem_u32(&b_full[sb]), pb);
            tc_fence_after();
            const uint32_t a_hi = tmem_a0 + (uint32_t)(st * 64);
            const uint32_t a_lo = a_hi + 32u;
            const uint64_t b_hi = make_smem_desc_sw128(smem_u32(smem_b + sb * C::kStageBBytes), 0, 1024);
            const uint64_t b_lo = make_smem_desc_sw128(smem_u32(smem_b + sb * C::kStageBBytes + C::kBBytes), 0, 1024);
#pragma unroll
            for (int k = 0; k < 4; ++k) {  // 4 x (K = 8 tf32) per 32-wide k-block
              const uint64_t o = (uint64_t)(k * 2);
              const uint32_t c = (uint32_t)(k * 8);
              umma_ts<true>(d, a_lo + c, b_hi + o, idesc, (kb | k) ? 1u : 0u);
              umma_ts<true>(d, a_hi + c, b_lo + o, idesc, 1u);
              umma_ts<true>(d, a_hi + c, b_hi + o, idesc, 1u);
            }
            umma_commit(smem_u32(&t_empty[st]));
            umma_commit(smem_u32(&b_empty[sb]));
            if (++st == C::kST) { st = 0; pt ^= 1; }
            if (++sb == C::kSB) { sb = 0; pb ^= 1; }
          }
          umma_commit(smem_u32(&acc_full[acc]));
          if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
      }
    }
  } else if (warp >= 4 && warp < 8) {
    // ===================== tf32 hi/lo split: shared memory -> registers -> TMEM =====================
    const int wq = warp & 3;
    const int row = wq * 32 + lane;                     // tile row == TMEM lane
    const uint32_t row_off = (uint32_t)row * 128u;
    const uint32_t sw = (uint32_t)(row & 7);
    const uint32_t lane_addr = (uint32_t)(wq * 32) << 16;
    int sa = 0, st = 0;
    uint32_t pa = 0, pt = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      for (int it = 0; it < p.n_nblk * p.total_kblocks; ++it) {
        mbar_wait(smem_u32(&a_full[sa]), pa);
        const uint32_t base = smem_u32(smem_a + sa * kABytes) + row_off;
        uint32_t hi[32], lo[32];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const uint4 v = lds128(base + ((((uint32_t)c) ^ sw) << 4));
          const uint32_t x[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint32_t h = x[j] & 0xffffe000u;
            hi[c * 4 + j] = h;
            lo[c * 4 + j] = __float_as_uint(__uint_as_float(x[j]) - __uint_as_float(h));
          }
        }
        mbar_wait(smem_u32(&t_empty[st]), pt ^ 1);
        tc_fence_after();
        const uint32_t ta = tmem_a0 + lane_addr + (uint32_t)(st * 64);
        tmem_st_32x32(ta, hi);
        tmem_st_32x32(ta + 32u, lo);
        // Release the landing slot only now: the stores above consume every loaded register, so the
        // LDS have COMPLETED.  Arriving right after the LDS were merely issued let the refill TMA
        // (async proxy) overtake a late shared-memory read: a few rows per 10^5 picked up the k-block
        // five stages ahead (tools/debug_proj.py signature test).
        mbar_arrive(smem_u32(&a_free[sa]));
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(smem_u32(&t_full[st]));
        if (++sa == C::kSA) { sa = 0; pa ^= 1; }
        if (++st == C::kST) { st = 0; pt ^= 1; }
      }
    }
  } else if (warp >= 8) {
    // ===================== epilogue: TMEM -> registers -> staging tile -> coalesced stores =====================
    const int wq = warp & 3;
    const uint32_t stg = smem_u32(smem_stage + wq * 4096);
    const uint32_t sw = (uint32_t)(lane & 7);
    int acc = 0;
    uint32_t acc_phase = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      for (int nb = 0; nb < p.n_nblk; ++nb) {
        mbar_wait(smem_u32(&acc_full[acc]), acc_phase);
        tc_fence_after();
        const long long row0 = tile * BM + wq * 32;
        const long long row = row0 + lane;
        const float rs = (row < p.n_rows && p.row_scale[nb]) ? __ldg(p.row_scale[nb] + row) : 1.f;
        const float* bias = p.bias[nb];
        float* outp = reinterpret_cast<float*>(p.out[nb]);
        const long long ld = p.ld_out[nb];
#pragma unroll 1
        for (int c = 0; c < BN / 32; ++c) {
          uint32_t r[32];
          tmem_ld_32x32(tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(acc * BN + c * 32), r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float f[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              float v = __uint_as_float(r[j * 4 + q]) * rs;
              if (bias) v += __ldg(bias + c * 32 + j * 4 + q);
              if (p.relu) v = fmaxf(v, 0.f);
              f[q] = v;
            }
            sts128(stg + (uint32_t)lane * 128u + ((((uint32_t)j) ^ sw) << 4),
                   make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]), __float_as_uint(f[3])));
          }
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int rr = i * 4 + (lane >> 3);            // row of the block, 8 lanes per row
            const uint32_t ch = (uint32_t)(lane & 7);
            const uint4 v = lds128(stg + (uint32_t)rr * 128u + ((ch ^ (uint32_t)(rr & 7)) << 4));
            if (row0 + rr < p.n_rows)
              *reinterpret_cast<uint4*>(outp + (row0 + rr) * ld + c * 32 + ch * 4) = v;
          }
          __syncwarp();
        }
        tc_fence_before();
        mbar_arrive(smem_u32(&acc_empty[acc]));
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, C::kTmemCols);
}

// ---- weight preparation: Bcat (alpha-scaled, concatenated along K or transposed), tf32 hi / lo ----
struct PrepArgs {
  const void* w[kMaxTerms];
  int k[kMaxTerms];
  float alpha[kMaxTerms];
  int n_terms, hidden, transpose, f32, split;
  void* b_hi;
  void* b_lo;
};
// forward  (transpose = 0): Bcat[h, koff_t + kk] = alpha_t * W_t[h, kk]          -> [hidden, sum k]
// backward (transpose = 1): Bcat[t * k_t + kk, h] = alpha_t * W_t[h, kk]         -> [sum k, hidden]
__global__ void prep_weights(const PrepArgs a) {
  int ktot = 0;
  for (int t = 0; t < a.n_terms; ++t) ktot += a.k[t];
  const int n = a.hidden * ktot;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int h = i / ktot;
    int kk = i % ktot, t = 0;
    while (kk >= a.k[t]) { kk -= a.k[t]; ++t; }
    const size_t src = (size_t)h * a.k[t] + kk;
    float v = a.f32 ? reinterpret_cast<const float*>(a.w[t])[src]
                    : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(a.w[t])[src]);
    v *= a.alpha[t];
    const size_t dst = a.transpose ? (size_t)(i % ktot) * a.hidden + h : (size_t)i;
    if (a.f32 && a.split) {
      const float hi = tf32_rna(v);
      reinterpret_cast<float*>(a.b_hi)[dst] = hi;
      reinterpret_cast<float*>(a.b_lo)[dst] = tf32_rna(v - hi);
    } else if (a.f32) {
      reinterpret_cast<float*>(a.b_hi)[dst] = v;
    } else {
      reinterpret_cast<__nv_bfloat16*>(a.b_hi)[dst] = __float2bfloat16_rn(v);
    }
  }
}

// ---- host ------------------------------------------------------------------------------------
EncodeTiledFn get_encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

int make_tmap_2d(CUtensorMap* map, const void* base, int dtype, uint64_t rows, uint64_t cols,
                 uint64_t ld_elems, uint32_t box_rows) {
  EncodeTiledFn enc = get_encode_tiled();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled entry point not available");
    return TRG_E_CUDA;
  }
  const int es = dtype == TRG_BF16 ? 2 : dtype == TRG_F8E4M3 ? 1 : 4;
  const CUtensorMapDataType dt = dtype == TRG_BF16     ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                 : dtype == TRG_F8E4M3 ? CU_TENSOR_MAP_DATA_TYPE_UINT8
                                                       : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {ld_elems * es};
  cuuint32_t box[2] = {(cuuint32_t)(128 / es), box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, dt, 2, const_cast<void*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(2d) failed: CUresult %d (rows=%llu cols=%llu ld=%llu box_rows=%u)",
              (int)r, (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld_elems,
              box_rows);
    return TRG_E_CUDA;
  }
  return TRG_OK;
}

template <bool F32, int BN>
int launch_cfg(const GemmParams& p, cudaStream_t st) {
  using C = Cfg<F32, BN>;
  static SmemAttrState attr;
  TRG_CUDA(ensure_dyn_smem(proj_tc_kernel<F32, BN>, C::kSmemBytes, attr));
  const long long n_tiles = (p.n_rows + BM - 1) / BM;
  const int grid = (int)std::min<long long>(n_tiles, grid_sms());
  proj_tc_kernel<F32, BN><<<grid, C::kThreads, C::kSmemBytes, st>>>(p);
  count_launch();
  TRG_LAUNCH_OK();
  return TRG_OK;
}

template <int BN>
int launch_cfg_a(const GemmParams& p, cudaStream_t st) {
  using C = CfgA<BN>;
  static SmemAttrState attr;
  TRG_CUDA(ensure_dyn_smem(proj_tc_f32a_kernel<BN>, C::kSmemBytes, attr));
  const long long n_tiles = (p.n_rows + BM - 1) / BM;
  const int grid = (int)std::min<long long>(n_tiles, grid_sms());
  proj_tc_f32a_kernel<BN><<<grid, C::kThreads, C::kSmemBytes, st>>>(p);
  count_launch();
  TRG_LAUNCH_OK();
  return TRG_OK;
}

static bool use_v1() { return debug_env_int("TRG_PROJ_V1", 0) == 1; }   // A/B, TRG_DEBUG builds only

int launch_gemm(const GemmParams& p, bool f32, int bn, cudaStream_t st) {
  if (f32 && !use_v1()) {       // split A operand in tensor memory (hidden <= 128: TMEM budget)
    if (bn == 64) return launch_cfg_a<64>(p, st);
    if (bn == 128) return launch_cfg_a<128>(p, st);
  }
  if (f32) {
    if (bn == 64) return launch_cfg<true, 64>(p, st);
    if (bn == 128) return launch_cfg<true, 128>(p, st);
    if (bn == 256) return launch_cfg<true, 256>(p, st);
  } else {
    if (bn == 64) return launch_cfg<false, 64>(p, st);
    if (bn == 128) return launch_cfg<false, 128>(p, st);
    if (bn == 256) return launch_cfg<false, 256>(p, st);
  }
  set_error("proj_tc: unsupported BN=%d", bn);
  return TRG_E_UNSUPPORTED;
}

size_t proj_tc_workspace_bytes(int ktot, int hidden, int dtype) {
  const size_t es = dtype == TRG_BF16 ? 2 : 4;
  return 2 * align_up((size_t)ktot * hidden * es, 1024);
}

bool proj_tc_eligible(const int* ks, int n_terms, int hidden, int dtype) {
  if (n_terms < 1 || n_terms > kMaxTerms) return false;
  if (hidden != 64 && hidden != 128 && hidden != 256) return false;
  const int kbe = dtype == TRG_BF16 ? 64 : 32;
  for (int i = 0; i < n_terms; ++i)
    if (ks[i] <= 0 || ks[i] % kbe != 0) return false;
  return get_encode_tiled() != nullptr;
}

// forward: out = act(sum_t alpha_t A_t W_t^T + bias)
int proj_tc_fwd(const trg_proj_term* terms, int n_terms, const float* bias, int64_t n_rows, int hidden,
                int dtype, int relu, void* out, void* ws, size_t ws_bytes, cudaStream_t st) {
  const bool f32 = dtype == TRG_F32;
  const int kbe = f32 ? 32 : 64;
  int ktot = 0;
  for (int i = 0; i < n_terms; ++i) ktot += terms[i].k;
  const size_t need = proj_tc_workspace_bytes(ktot, hidden, dtype);
  if (!ws || ws_bytes < need) {
    set_error("trg_sage_proj_fwd: workspace %zu < required %zu", ws_bytes, need);
    return TRG_E_WORKSPACE;
  }
  PrepArgs pa{};
  for (int i = 0; i < n_terms; ++i) { pa.w[i] = terms[i].w; pa.k[i] = terms[i].k; pa.alpha[i] = terms[i].alpha; }
  pa.n_terms = n_terms; pa.hidden = hidden; pa.transpose = 0; pa.f32 = f32; pa.split = 1;
  pa.b_hi = ws;
  pa.b_lo = reinterpret_cast<char*>(ws) + need / 2;
  prep_weights<<<std::min(64, (hidden * ktot + 255) / 256), 256, 0, st>>>(pa);
  count_launch();
  TRG_LAUNCH_OK();

  GemmParams p{};
  for (int i = 0; i < n_terms; ++i) {
    int rc = make_tmap_2d(&p.a_map[i], terms[i].a, dtype, (uint64_t)n_rows, terms[i].k, terms[i].k, BM);
    if (rc) return rc;
    p.a_kblocks[i] = terms[i].k / kbe;
  }
  int rc = make_tmap_2d(&p.b_hi_map, pa.b_hi, dtype, hidden, ktot, ktot, hidden);
  if (rc) return rc;
  if (f32) {
    rc = make_tmap_2d(&p.b_lo_map, pa.b_lo, dtype, hidden, ktot, ktot, hidden);
    if (rc) return rc;
  }
  p.n_a = n_terms; p.n_nblk = 1; p.total_kblocks = ktot / kbe; p.relu = relu; p.n_rows = n_rows;
  p.out[0] = out; p.ld_out[0] = hidden; p.row_scale[0] = nullptr; p.bias[0] = bias;
  return launch_gemm(p, f32, hidden, st);
}

// backward w.r.t. inputs: d_a_t = row_scale_t * (alpha_t * dZ @ W_t), one n-block per term
int proj_tc_bwd_input(const void* dz, const trg_proj_bwd_term* terms, int n_terms, int64_t n_rows,
                      int hidden, int dtype, void* ws, size_t ws_bytes, cudaStream_t st) {
  const bool f32 = dtype == TRG_F32;
  const int kbe = f32 ? 32 : 64;
  const int bn = terms[0].k;
  int ktot = 0;
  for (int i = 0; i < n_terms; ++i) ktot += terms[i].k;
  const size_t need = proj_tc_workspace_bytes(ktot, hidden, dtype);
  if (!ws || ws_bytes < need) {
    set_error("trg_sage_proj_bwd_input: workspace %zu < required %zu", ws_bytes, need);
    return TRG_E_WORKSPACE;
  }
  PrepArgs pa{};
  for (int i = 0; i < n_terms; ++i) { pa.w[i] = terms[i].w; pa.k[i] = terms[i].k; pa.alpha[i] = terms[i].alpha; }
  pa.n_terms = n_terms; pa.hidden = hidden; pa.transpose = 1; pa.f32 = f32; pa.split = 1;
  pa.b_hi = ws;
  pa.b_lo = reinterpret_cast<char*>(ws) + need / 2;
  prep_weights<<<std::min(64, (hidden * ktot + 255) / 256), 256, 0, st>>>(pa);
  count_launch();
  TRG_LAUNCH_OK();

  GemmParams p{};
  int rc = make_tmap_2d(&p.a_map[0], dz, dtype, (uint64_t)n_rows, hidden, hidden, BM);
  if (rc) return rc;
  p.a_kblocks[0] = hidden / kbe;
  rc = make_tmap_2d(&p.b_hi_map, pa.b_hi, dtype, ktot, hidden, hidden, bn);
  if (rc) return rc;
  if (f32) {
    rc = make_tmap_2d(&p.b_lo_map, pa.b_lo, dtype, ktot, hidden, hidden, bn);
    if (rc) return rc;
  }
  p.n_a = 1; p.n_nblk = n_terms; p.total_kblocks = hidden / kbe; p.relu = 0; p.n_rows = n_rows;
  for (int i = 0; i < n_terms; ++i) {
    p.out[i] = terms[i].d_a; p.ld_out[i] = terms[i].k; p.row_scale[i] = terms[i].row_scale;
    p.bias[i] = nullptr;
  }
  return launch_gemm(p, f32, bn, st);
}

// Shape-generic fallback for the input gradient: transposed alpha-scaled weights, then the SIMT GEMM.
int proj_simt_bwd_input(const void* dz, const trg_proj_bwd_term* terms, int n_terms, int64_t n_rows,
                        int hidden, int dtype, void* ws, size_t ws_bytes, cudaStream_t st) {
  int ktot = 0;
  for (int i = 0; i < n_terms; ++i) ktot += terms[i].k;
  const size_t need = proj_tc_workspace_bytes(ktot, hidden, dtype);
  if (!ws || ws_bytes < need) {
    set_error("trg_sage_proj_bwd_input: workspace %zu < required %zu", ws_bytes, need);
    return TRG_E_WORKSPACE;
  }
  PrepArgs pa{};
  for (int i = 0; i < n_terms; ++i) { pa.w[i] = terms[i].w; pa.k[i] = terms[i].k; pa.alpha[i] = terms[i].alpha; }
  pa.n_terms = n_terms; pa.hidden = hidden; pa.transpose = 1; pa.f32 = dtype == TRG_F32; pa.split = 0;
  pa.b_hi = ws; pa.b_lo = nullptr;
  prep_weights<<<std::min(64, (hidden * ktot + 255) / 256), 256, 0, st>>>(pa);
  count_launch();
  TRG_LAUNCH_OK();
  const size_t es = dtype == TRG_BF16 ? 2 : 4;
  int koff = 0;
  for (int i = 0; i < n_terms; ++i) {
    trg_proj_term t{dz, reinterpret_cast<char*>(ws) + (size_t)koff * hidden * es, hidden, 1.0f};
    int rc = proj_simt_launch(&t, 1, nullptr, terms[i].row_scale, n_rows, terms[i].k, dtype, 0,
                              terms[i].d_a, st);
    if (rc) return rc;
    koff += terms[i].k;
  }
  return TRG_OK;
}

}  // namespace tc
}  // namespace trg
