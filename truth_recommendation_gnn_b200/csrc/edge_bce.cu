// K4 -- fused positive/negative edge scoring + BCE-with-logits, forward and (user side) backward.
//
// Replaces train_gnn.py:259-281 (four [E,H] gathers, two mul+rowsum, two BCEWithLogitsLoss) and
// the index_put_(accumulate=True) half of loss.backward() (train_gnn.py:283) that lands on
// user_emb.  Positive edges arrive grouped by user (CSR keyed on pos_u), so the user row is
// read ONCE per user instead of twice per edge, dloss/du is produced in the same pass without
// atomics, and per-edge coefficients c_pos/c_neg are left for the post-side gather passes
// (trg_gather_wsum).  HBM-bound: 2 random post rows per edge.
#include <cstdlib>

#include "common.cuh"

namespace trg {
namespace {

constexpr int kThreads = 256;

struct BceArgs {
  const int* rowptr;
  const int* col_p;
  const int* eid;
  const long long* neg_p;
  const void* u;
  const void* p;
  const float* wbar;
  float* c_pos;
  float* c_neg;
  void* g_u;
  double* partials;  // [gridDim.x][2]
  int64_t n_users;
  float inv_e;
  int row_vecs;
  int label;        // single-row mode: 1 = positives (softplus(-x), weight wbar), 0 = negatives
  int accumulate;   // single-row mode: add to the existing anchor-gradient rows
  int relu_gate;    // single-row mode: zero the anchor gradient where the anchor row is <= 0 (the anchor
                    // table is a ReLU output: this is the ReLU derivative, fused into the final write)
};

__device__ __forceinline__ float softplus(float x) {  // log(1 + e^x), stable
  return fmaxf(x, 0.f) + log1pf(expf(-fabsf(x)));
}
__device__ __forceinline__ float sigmoid(float x) {
  const float e = expf(-fabsf(x));
  return x >= 0.f ? __fdiv_rn(1.f, 1.f + e) : __fdiv_rn(e, 1.f + e);
}

// Each group of LPR lanes owns R consecutive users and walks their positive edges as one continuous
// stream (same scheme as gather_reduce_seg): the (post id, edge id) pairs of the next 32-edge chunk
// and the dependent neg_p[eid] lookup are prefetched two chunks / one chunk ahead, so the only
// exposed latency is that of the post rows themselves (2 per edge, kUnroll edges in flight).
//
// TWO = true : anchor rows = users, two gathered post rows per edge (positive + sampled negative):
//              the single-GPU fused loss.
// TWO = false: one gathered row per edge and a label per launch: the multi-GPU form, where the loss is
//              evaluated by the OWNER OF THE POST (anchor rows = local posts, gathered rows = the
//              all-gathered user table, which is 5x smaller than the post table).
template <typename T, int LPR, int VPL, int R, bool TWO>
__global__ void __launch_bounds__(kThreads, VPL == 1 ? 3 : 2) edge_bce(const BceArgs a) {
  constexpr int kVec = Elem<T>::kVec;
  constexpr int kUnroll = (LPR < 8 ? (LPR >= 4 ? 2 : 1) : (VPL == 1 ? 4 : 2)) * (TWO ? 1 : 2);
  static_assert(R < LPR, "row boundaries are held one per lane");
  __shared__ double red[2][kThreads / 32];
  // fp64 running sums of this thread's fp32 loss terms, folded in once per chunk: one row group may walk a
  // hub row of millions of edges, whose terms a single fp32 sum would carry ~1e-4 off
  __shared__ double lane_sum[2][kThreads];
  const int lane = threadIdx.x & 31;
  const int gl = lane & (LPR - 1);
  const unsigned gmask = LPR == 32 ? 0xffffffffu : (((1u << LPR) - 1u) << (lane & ~(LPR - 1)));
  const int64_t r0 = ((int64_t)blockIdx.x * (kThreads / LPR) + threadIdx.x / LPR) * R;
  const bool want_grad = a.g_u != nullptr;
  float sp_sum = 0.f, sn_sum = 0.f;
  lane_sum[0][threadIdx.x] = lane_sum[1][threadIdx.x] = 0.0;   // thread-private slots: no barrier

  if (r0 < a.n_users) {
    const int nr = (int)((a.n_users - r0) < (int64_t)R ? (a.n_users - r0) : (int64_t)R);
    const int my_ptr = ldg_stream(a.rowptr + r0 + min(gl, nr));
    const int e_end = __shfl_sync(gmask, my_ptr, nr, LPR);
    int e0 = __shfl_sync(gmask, my_ptr, 0, LPR);
    const size_t row_bytes = (size_t)a.row_vecs * 16;
    const char* pb = reinterpret_cast<const char*>(a.p);
    const char* ub = reinterpret_cast<const char*>(a.u);
    const float wbar = __ldg(a.wbar);

    bool act[VPL];
    float uf[VPL][kVec], ga[VPL][kVec];
    uint4 u_nxt[VPL];
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      act[i] = gl + i * LPR < a.row_vecs;
#pragma unroll
      for (int k = 0; k < kVec; ++k) uf[i][k] = ga[i][k] = 0.f;
      u_nxt[i] = make_uint4(0, 0, 0, 0);
      if (act[i]) {
        Elem<T>::unpack(ldg_row(ub + (size_t)r0 * row_bytes + (size_t)(gl + i * LPR) * 16), uf[i]);
        if (nr > 1) u_nxt[i] = ldg_row(ub + (size_t)(r0 + 1) * row_bytes + (size_t)(gl + i * LPR) * 16);
      }
    }
    int cur = 0;
    int cur_end = __shfl_sync(gmask, my_ptr, 1, LPR);

    auto flush = [&]() {   // close user row `cur`: write dL/du, move to the next user's row
      if (want_grad) {
        char* ob = reinterpret_cast<char*>(a.g_u) + (size_t)(r0 + cur) * row_bytes;
#pragma unroll
        for (int i = 0; i < VPL; ++i)
          if (act[i]) {
            if (!TWO && a.accumulate) {
              float f[kVec];
              Elem<T>::unpack(*reinterpret_cast<const uint4*>(ob + (size_t)(gl + i * LPR) * 16), f);
#pragma unroll
              for (int k = 0; k < kVec; ++k) ga[i][k] += f[k];
            }
            if (!TWO && a.relu_gate) {
#pragma unroll
              for (int k = 0; k < kVec; ++k) ga[i][k] = uf[i][k] > 0.f ? ga[i][k] : 0.f;
            }
            stg_stream(ob + (size_t)(gl + i * LPR) * 16, Elem<T>::pack(ga[i]));
          }
      }
      ++cur;
      cur_end = __shfl_sync(gmask, my_ptr, min(cur + 1, nr), LPR);
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        Elem<T>::unpack(u_nxt[i], uf[i]);
#pragma unroll
        for (int k = 0; k < kVec; ++k) ga[i][k] = 0.f;
        if (act[i] && cur + 1 < nr)
          u_nxt[i] = ldg_row(ub + (size_t)(r0 + cur + 1) * row_bytes + (size_t)(gl + i * LPR) * 16);
      }
    };

    auto load_idx = [&](int e, int& cp, int& id) {
      cp = 0; id = 0;
      if (e < e_end) {
        cp = ldg_stream(a.col_p + e);
        id = a.eid ? ldg_stream(a.eid + e) : e;   // eid == NULL: coefficients are written in CSR edge order
      }
    };
    // index pipeline: (post id, edge id) two chunks ahead, the dependent neg_p[edge id] one ahead.
    // (A bulk L2 prefetch of the next chunk's rows was measured SLOWER: 13.5 vs 12.7 ms at cfg 2.)
    int cp_cur, id_cur, cn_cur = 0, cp_nxt, id_nxt;
    load_idx(e0 + gl, cp_cur, id_cur);
    if (TWO && e0 + gl < e_end) cn_cur = (int)ldg_stream(a.neg_p + id_cur);
    load_idx(e0 + LPR + gl, cp_nxt, id_nxt);

    while (e0 < e_end) {
      const int cnt = min(LPR, e_end - e0);
      int cn_nxt = 0;
      if (TWO && e0 + LPR + gl < e_end) cn_nxt = (int)ldg_stream(a.neg_p + id_nxt);
      int cp_nn, id_nn;
      load_idx(e0 + 2 * LPR + gl, cp_nn, id_nn);
      float my_cpos = 0.f, my_cneg = 0.f;

      int t = 0;
      while (t < cnt) {
        while (e0 + t >= cur_end) flush();               // group-uniform: next user's row
        // a batch never straddles a user boundary: every edge in it is scored against uf
        const int bsz = min(min(kUnroll, cnt - t), cur_end - (e0 + t));
        uint4 vp[kUnroll][VPL], vn[kUnroll][VPL];
#pragma unroll
        for (int q = 0; q < kUnroll; ++q) {
          const int cpq = __shfl_sync(gmask, cp_cur, t + q, LPR);
          const int cnq = __shfl_sync(gmask, cn_cur, t + q, LPR);
          if (q < bsz) {
#pragma unroll
            for (int i = 0; i < VPL; ++i)
              if (act[i]) {
                vp[q][i] = ldg_row(pb + (size_t)cpq * row_bytes + (size_t)(gl + i * LPR) * 16);
                if (TWO) vn[q][i] = ldg_row(pb + (size_t)cnq * row_bytes + (size_t)(gl + i * LPR) * 16);
              }
          }
        }
        // partial dots, then ONE halving butterfly over the group: afterwards each lane holds the
        // group total of one of the 2*kUnroll scores (value j on lanes [j*LPR/NV, (j+1)*LPR/NV))
        constexpr int NV = TWO ? 2 * kUnroll : kUnroll;
        static_assert(LPR >= NV, "transpose-reduce needs at least one lane per value");
        float v[NV];
#pragma unroll
        for (int q = 0; q < kUnroll; ++q) {
          float dp = 0.f, dn = 0.f;
          if (q < bsz) {
#pragma unroll
            for (int i = 0; i < VPL; ++i) {
              if (act[i]) {
                float fp[kVec], fn[kVec];
                Elem<T>::unpack(vp[q][i], fp);
                if (TWO) Elem<T>::unpack(vn[q][i], fn);
#pragma unroll
                for (int k = 0; k < kVec; ++k) {
                  dp = fmaf(uf[i][k], fp[k], dp);
                  if (TWO) dn = fmaf(uf[i][k], fn[k], dn);
                }
              }
            }
          }
          if (TWO) {
            v[2 * q] = dp;
            v[2 * q + 1] = dn;
          } else {
            v[q] = dp;
          }
        }
        int nv = NV;
#pragma unroll
        for (int o = LPR / 2; o > 0; o >>= 1) {
          if (nv > 1) {
            nv >>= 1;
#pragma unroll
            for (int i = 0; i < NV / 2; ++i) {
              if (i < nv) {
                const bool hi = (gl & o) != 0;
                const float send = hi ? v[i] : v[i + nv];
                const float keep = hi ? v[i + nv] : v[i];
                v[i] = keep + __shfl_xor_sync(gmask, send, o, LPR);
              }
            }
          } else {
            v[0] += __shfl_xor_sync(gmask, v[0], o, LPR);
          }
        }
        constexpr int kLanesPerVal = LPR / NV;
        const int j = gl / kLanesPerVal;                 // the score this lane finishes
        const bool is_neg = TWO ? (j & 1) : (a.label == 0);
        const float z = is_neg ? v[0] : -v[0];           // loss term = softplus(z)
        const float spv = softplus(z);
        if ((gl % kLanesPerVal) == 0 && (TWO ? (j >> 1) : j) < bsz) {
          if (is_neg) sn_sum += spv; else sp_sum += spv;
        }
        if (want_grad) {
          const float coef = (is_neg ? 1.f : -wbar) * sigmoid(z) * a.inv_e;
#pragma unroll
          for (int q = 0; q < kUnroll; ++q) {
            const float cpos = __shfl_sync(gmask, coef, (TWO ? 2 * q : q) * kLanesPerVal, LPR);
            const float cneg = TWO ? __shfl_sync(gmask, coef, (2 * q + 1) * kLanesPerVal, LPR) : 0.f;
            if (q < bsz) {
              if (gl == t + q) {
                my_cpos = cpos;
                my_cneg = cneg;
              }
#pragma unroll
              for (int i = 0; i < VPL; ++i)
                if (act[i]) {
                  float fp[kVec], fn[kVec];
                  Elem<T>::unpack(vp[q][i], fp);
                  if (TWO) Elem<T>::unpack(vn[q][i], fn);
#pragma unroll
                  for (int k = 0; k < kVec; ++k)
                    ga[i][k] = TWO ? fmaf(cpos, fp[k], fmaf(cneg, fn[k], ga[i][k])) : fmaf(cpos, fp[k], ga[i][k]);
                }
            }
          }
        }
        t += bsz;
      }
      if (want_grad && e0 + gl < e_end) {
        a.c_pos[id_cur] = my_cpos;
        if (TWO) a.c_neg[id_cur] = my_cneg;
      }
      lane_sum[0][threadIdx.x] += (double)sp_sum;
      lane_sum[1][threadIdx.x] += (double)sn_sum;
      sp_sum = sn_sum = 0.f;
      e0 += LPR;
      cp_cur = cp_nxt; id_cur = id_nxt; cn_cur = cn_nxt;
      cp_nxt = cp_nn; id_nxt = id_nn;
    }
    while (cur < nr) flush();
  }

  // deterministic CTA reduction -> one (sp, sn) pair of doubles per CTA
  double dsp = lane_sum[0][threadIdx.x], dsn = lane_sum[1][threadIdx.x];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    dsp += __shfl_xor_sync(0xffffffffu, dsp, o);
    dsn += __shfl_xor_sync(0xffffffffu, dsn, o);
  }
  if (lane == 0) {
    red[0][threadIdx.x >> 5] = dsp;
    red[1][threadIdx.x >> 5] = dsn;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double s0 = 0, s1 = 0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) {
      s0 += red[0][w];
      s1 += red[1][w];
    }
    a.partials[2 * (size_t)blockIdx.x] = s0;
    a.partials[2 * (size_t)blockIdx.x + 1] = s1;
  }
}

// Single-row form for 512-byte rows (fp32 H = 128, bf16 H = 256), gathered rows staged through a
// per-warp cp.async ring.  ncu on the register form above: 5.0 TB/s of DRAM traffic, long-scoreboard
// stalls -- a warp has its 8 row loads in flight only until they land, then reduces / exponentiates /
// accumulates with nothing outstanding, and 80 registers cap the SM at 24 warps.  Here the row loads do
// not occupy registers: every warp keeps two 8-edge groups (8 KB) in flight in shared memory while it
// works on a third, so 8-16 row loads per warp are outstanding during the arithmetic as well.
// Same arithmetic in the same order as edge_bce<T, 32, 1, 4, false>: results are bit-identical.
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ uint4 lds128_bce(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}

constexpr int kRingG = 8;                      // edges per cp.async group
constexpr int kRingS = 16;                     // ring slots per warp (two groups)
constexpr int kRingBytes = (kThreads / 32) * kRingS * 512;

template <typename T>
__global__ void __launch_bounds__(kThreads, 3) edge_anchor_ring(const BceArgs a) {
  constexpr int kVec = Elem<T>::kVec;
  constexpr int R = 4, G = kRingG, S = kRingS;
  constexpr unsigned full = 0xffffffffu;
  extern __shared__ __align__(16) unsigned char ring_raw[];
  __shared__ double red[2][kThreads / 32];
  __shared__ double lane_sum[kThreads];   // fp64 running sum of the thread's fp32 loss terms (as in edge_bce)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t ring_a = static_cast<uint32_t>(__cvta_generic_to_shared(ring_raw)) +
                          (uint32_t)(warp * S * 512 + lane * 16);
  const int64_t r0 = ((int64_t)blockIdx.x * (kThreads / 32) + warp) * R;
  const bool want_grad = a.g_u != nullptr;
  float s_sum = 0.f;
  lane_sum[threadIdx.x] = 0.0;

  if (r0 < a.n_users) {
    const int nr = (int)((a.n_users - r0) < (int64_t)R ? (a.n_users - r0) : (int64_t)R);
    const int my_ptr = ldg_stream(a.rowptr + r0 + min(lane, nr));
    const int e_end = __shfl_sync(full, my_ptr, nr);
    const int e_beg = __shfl_sync(full, my_ptr, 0);
    const char* pb = reinterpret_cast<const char*>(a.p);
    const char* ub = reinterpret_cast<const char*>(a.u);
    const float wbar = __ldg(a.wbar);
    const bool is_neg = a.label == 0;

    float uf[kVec], ga[kVec];
    uint4 u_nxt = make_uint4(0, 0, 0, 0);
#pragma unroll
    for (int k = 0; k < kVec; ++k) ga[k] = 0.f;
    Elem<T>::unpack(ldg_row(ub + (size_t)r0 * 512 + (size_t)lane * 16), uf);
    if (nr > 1) u_nxt = ldg_row(ub + (size_t)(r0 + 1) * 512 + (size_t)lane * 16);
    int cur = 0;
    int cur_end = __shfl_sync(full, my_ptr, 1);

    auto flush = [&]() {   // close anchor row `cur`: write its gradient, move to the next row
      if (want_grad) {
        char* ob = reinterpret_cast<char*>(a.g_u) + (size_t)(r0 + cur) * 512 + (size_t)lane * 16;
        if (a.accumulate) {
          float f[kVec];
          Elem<T>::unpack(*reinterpret_cast<const uint4*>(ob), f);
#pragma unroll
          for (int k = 0; k < kVec; ++k) ga[k] += f[k];
        }
        if (a.relu_gate) {
#pragma unroll
          for (int k = 0; k < kVec; ++k) ga[k] = uf[k] > 0.f ? ga[k] : 0.f;
        }
        stg_stream(ob, Elem<T>::pack(ga));
      }
      ++cur;
      cur_end = __shfl_sync(full, my_ptr, min(cur + 1, nr));
      Elem<T>::unpack(u_nxt, uf);
#pragma unroll
      for (int k = 0; k < kVec; ++k) ga[k] = 0.f;
      if (cur + 1 < nr) u_nxt = ldg_row(ub + (size_t)(r0 + cur + 1) * 512 + (size_t)lane * 16);
    };
    auto load_id = [&](int ebase) -> int {          // lane l < G: gathered-row id of edge ebase + l
      const int e = ebase + lane;
      return (lane < G && e < e_end) ? ldg_stream(a.col_p + e) : 0;
    };
    auto issue = [&](int ebase, int ids, int slot0) {   // one cp.async group: rows of edges ebase .. ebase+G-1
#pragma unroll
      for (int q = 0; q < G; ++q) {
        const int rid = __shfl_sync(full, ids, q);
        if (ebase + q < e_end)
          cp_async16(ring_a + (uint32_t)(((slot0 + q) & (S - 1)) * 512), pb + (size_t)rid * 512 + (size_t)lane * 16);
      }
      cp_async_commit();
    };

    {
      const int id0 = load_id(e_beg), id1 = load_id(e_beg + G);
      issue(e_beg, id0, 0);
      issue(e_beg + G, id1, G);
    }
    int nid = load_id(e_beg + 2 * G);   // ids of the group issued at the end of the current iteration
    int slot = 0;
    for (int e_base = e_beg; e_base < e_end; e_base += G) {
      const int cnt = min(G, e_end - e_base);
      int my_id = 0;
      if (want_grad && lane < cnt) my_id = a.eid ? ldg_stream(a.eid + e_base + lane) : e_base + lane;
      cp_async_wait<1>();     // this group has landed (the next one may still be in flight)
      __syncwarp();
      float my_c = 0.f;
      int t = 0;
      while (t < cnt) {
        while (e_base + t >= cur_end) flush();               // warp-uniform: next anchor row
        const int bsz = min(cnt - t, cur_end - (e_base + t));   // a batch never straddles a row boundary
        uint4 vp[G];
        float v[G];
#pragma unroll
        for (int q = 0; q < G; ++q) {
          float dp = 0.f;
          if (q < bsz) {
            vp[q] = lds128_bce(ring_a + (uint32_t)(((slot + t + q) & (S - 1)) * 512));
            float fp[kVec];
            Elem<T>::unpack(vp[q], fp);
#pragma unroll
            for (int k = 0; k < kVec; ++k) dp = fmaf(uf[k], fp[k], dp);
          }
          v[q] = dp;
        }
        // halving butterfly: afterwards lanes [4 j, 4 j + 4) hold the warp total of score j
        int nv = G;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          if (nv > 1) {
            nv >>= 1;
#pragma unroll
            for (int i = 0; i < G / 2; ++i) {
              if (i < nv) {
                const bool hi = (lane & o) != 0;
                const float send = hi ? v[i] : v[i + nv];
                const float keep = hi ? v[i + nv] : v[i];
                v[i] = keep + __shfl_xor_sync(full, send, o);
              }
            }
          } else {
            v[0] += __shfl_xor_sync(full, v[0], o);
          }
        }
        constexpr int kLanesPerVal = 32 / G;
        const int j = lane / kLanesPerVal;
        const float z = is_neg ? v[0] : -v[0];           // loss term = softplus(z)
        const float spv = softplus(z);
        if ((lane % kLanesPerVal) == 0 && j < bsz) s_sum += spv;
        if (want_grad) {
          const float coef = (is_neg ? 1.f : -wbar) * sigmoid(z) * a.inv_e;
#pragma unroll
          for (int q = 0; q < G; ++q) {
            const float cq = __shfl_sync(full, coef, q * kLanesPerVal);
            if (q < bsz) {
              if (lane == t + q) my_c = cq;
              float fp[kVec];
              Elem<T>::unpack(vp[q], fp);
#pragma unroll
              for (int k = 0; k < kVec; ++k) ga[k] = fmaf(cq, fp[k], ga[k]);
            }
          }
        }
        t += bsz;
      }
      if (want_grad && lane < cnt) a.c_pos[my_id] = my_c;
      lane_sum[threadIdx.x] += (double)s_sum;
      s_sum = 0.f;
      __syncwarp();           // every lane is done with this group's slots: refill them two groups ahead
      const int nid_next = load_id(e_base + 3 * G);
      issue(e_base + 2 * G, nid, slot);
      nid = nid_next;
      slot = (slot + G) & (S - 1);
    }
    while (cur < nr) flush();                               // last row and trailing empty rows
    cp_async_wait<0>();
  }

  // deterministic CTA reduction -> one (sp, sn) pair of doubles per CTA (layout of edge_bce)
  double dsum = lane_sum[threadIdx.x];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) dsum += __shfl_xor_sync(0xffffffffu, dsum, o);
  if (lane == 0) red[0][warp] = dsum;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s0 = 0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) s0 += red[0][w];
    const bool neg = a.label == 0;
    a.partials[2 * (size_t)blockIdx.x] = neg ? 0.0 : s0;
    a.partials[2 * (size_t)blockIdx.x + 1] = neg ? s0 : 0.0;
  }
}

// Fixed-order final reduction: loss = wbar * mean(softplus(-pos)) + mean(softplus(neg)).
__global__ void __launch_bounds__(1024) edge_bce_finish(const double* __restrict__ partials,
                                                        int64_t n_parts, const float* wbar,
                                                        double n_edges, float* loss_out) {
  __shared__ double red[2][32];
  double s0 = 0, s1 = 0;
  for (int64_t i = threadIdx.x; i < n_parts; i += 1024) {
    s0 += partials[2 * i];
    s1 += partials[2 * i + 1];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s0 += __shfl_xor_sync(0xffffffffu, s0, o);
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
  }
  if ((threadIdx.x & 31) == 0) {
    red[0][threadIdx.x >> 5] = s0;
    red[1][threadIdx.x >> 5] = s1;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    s0 = s1 = 0;
    for (int w = 0; w < 32; ++w) {
      s0 += red[0][w];
      s1 += red[1][w];
    }
    const float pos_loss = (float)(s0 / n_edges);  // 0/0 = NaN for E = 0, like torch's mean
    const float neg_loss = (float)(s1 / n_edges);
    loss_out[0] = __ldg(wbar) * pos_loss + neg_loss;
  }
}

template <typename T, bool TWO>
int launch_bce(BceArgs& a, int64_t* n_blocks_out, cudaStream_t st, bool dry) {
  const int rv = a.row_vecs;
#define TRG_BCE_CASE(LPR, VPL, R)                                                     \
  {                                                                                   \
    const int64_t grid = ceil_div<int64_t>(a.n_users, (int64_t)(kThreads / LPR) * R); \
    *n_blocks_out = grid;                                                             \
    if (!dry) edge_bce<T, LPR, VPL, R, TWO><<<(unsigned)grid, kThreads, 0, st>>>(a);  \
  }
  if (rv <= 2) TRG_BCE_CASE(2, 1, 1)
  else if (rv <= 4) TRG_BCE_CASE(4, 1, 2)
  else if (rv <= 8) TRG_BCE_CASE(8, 1, 4)
  else if (rv <= 16) TRG_BCE_CASE(16, 1, 4)
  else if (rv <= 32) TRG_BCE_CASE(32, 1, 4)
  else if (rv <= 64) TRG_BCE_CASE(32, 2, 4)
  else {
    set_error("trg_edge_bce_fwd: rows wider than 1024 bytes are not supported (row_vecs=%d)", rv);
    return TRG_E_UNSUPPORTED;
  }
#undef TRG_BCE_CASE
  return TRG_OK;
}

}  // namespace
}  // namespace trg

using namespace trg;

// A/B switch (TRG_DEBUG builds only): TRG_K4_RING=0 keeps the register form
static bool anchor_ring_off() { return debug_env_int("TRG_K4_RING", 1) == 0; }

extern "C" size_t trg_edge_bce_workspace_bytes(int64_t n_users) {
  if (n_users < 0) return 0;
  // worst case: one warp per user -> 8 users per CTA, 2 doubles per CTA
  return align_up((size_t)(ceil_div<int64_t>(n_users, 8) + 1) * 16, 256);
}

extern "C" int trg_edge_bce_fwd(const int32_t* rowptr_u, const int32_t* col_p, const int32_t* eid,
                                const int64_t* neg_p, const void* u, const void* p, int64_t n_users,
                                int64_t n_edges, int32_t hidden, int dtype, const float* wbar,
                                float* loss_out, float* c_pos, float* c_neg, void* g_u,
                                void* workspace, size_t workspace_bytes, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  TRG_CHECK_ARG(n_users >= 0 && n_edges >= 0, "trg_edge_bce_fwd: negative size");
  TRG_CHECK_ARG(loss_out && wbar, "trg_edge_bce_fwd: NULL loss_out/wbar");
  TRG_CHECK_ARG((c_pos == nullptr) == (g_u == nullptr) && (c_neg == nullptr) == (g_u == nullptr),
                "trg_edge_bce_fwd: c_pos, c_neg and g_u must be all NULL or all non-NULL");
  TRG_CHECK_ARG(n_users == 0 || (rowptr_u && u && p), "trg_edge_bce_fwd: NULL rowptr / tables");
  TRG_CHECK_ARG(((uintptr_t)u | (uintptr_t)p | (uintptr_t)g_u) % 16 == 0,
                "trg_edge_bce_fwd: tables must be 16-byte aligned");
  const int es = dtype == TRG_BF16 ? 2 : 4;
  TRG_CHECK_ARG(dtype == TRG_F32 || dtype == TRG_BF16, "trg_edge_bce_fwd: unknown dtype %d", dtype);
  TRG_CHECK_ARG(hidden > 0 && (hidden * es) % 16 == 0,
                "trg_edge_bce_fwd: row width %d x %d bytes is not a multiple of 16 bytes", hidden, es);
  if ((int64_t)hidden * es > 1024) {   // checked here, not at dispatch, so n_users = 0 is refused alike
    set_error("trg_edge_bce_fwd: rows wider than 1024 bytes are not supported (%d x %d bytes)", hidden, es);
    return TRG_E_UNSUPPORTED;
  }
  if (workspace == nullptr || workspace_bytes < trg_edge_bce_workspace_bytes(n_users)) {
    set_error("trg_edge_bce_fwd: workspace %zu < required %zu", workspace_bytes,
              trg_edge_bce_workspace_bytes(n_users));
    return TRG_E_WORKSPACE;
  }
  BceArgs a{};
  a.rowptr = rowptr_u; a.col_p = col_p; a.eid = eid; a.neg_p = (const long long*)neg_p;
  a.u = u; a.p = p; a.wbar = wbar; a.c_pos = c_pos; a.c_neg = c_neg; a.g_u = g_u;
  a.partials = reinterpret_cast<double*>(workspace);
  a.n_users = n_users;
  a.inv_e = n_edges > 0 ? (float)(1.0 / (double)n_edges) : 0.f;
  a.row_vecs = hidden * es / 16;
  int64_t n_blocks = 0;
  if (n_users > 0) {
    int rc = dtype == TRG_F32 ? launch_bce<float, true>(a, &n_blocks, st, false)
                              : launch_bce<__nv_bfloat16, true>(a, &n_blocks, st, false);
    if (rc) return rc;
    count_launch();
    TRG_LAUNCH_OK();
  }
  edge_bce_finish<<<1, 1024, 0, st>>>(a.partials, n_blocks, wbar, (double)n_edges, loss_out);
  count_launch();
  TRG_LAUNCH_OK();
  return TRG_OK;
}

extern "C" int trg_edge_anchor_loss(const int32_t* rowptr, const int32_t* col, const int32_t* eid,
                                    const void* anchor, const void* gathered, int64_t n_rows,
                                    int64_t n_edges_scale, int32_t hidden, int dtype, int label,
                                    const float* wbar, float* loss_out, float* coef_out, void* g_anchor,
                                    int accumulate, int relu_gate, void* workspace, size_t workspace_bytes,
                                    void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  TRG_CHECK_ARG(n_rows >= 0 && n_edges_scale >= 0, "trg_edge_anchor_loss: negative size");
  TRG_CHECK_ARG(loss_out && wbar, "trg_edge_anchor_loss: NULL loss_out/wbar");
  TRG_CHECK_ARG((coef_out == nullptr) == (g_anchor == nullptr),
                "trg_edge_anchor_loss: coef_out and g_anchor must be both NULL or both non-NULL");
  TRG_CHECK_ARG(n_rows == 0 || (rowptr && anchor), "trg_edge_anchor_loss: NULL rowptr / anchor table");
  TRG_CHECK_ARG(((uintptr_t)anchor | (uintptr_t)gathered | (uintptr_t)g_anchor) % 16 == 0,
                "trg_edge_anchor_loss: tables must be 16-byte aligned");
  TRG_CHECK_ARG(dtype == TRG_F32 || dtype == TRG_BF16, "trg_edge_anchor_loss: unknown dtype %d", dtype);
  const int es = dtype == TRG_BF16 ? 2 : 4;
  TRG_CHECK_ARG(hidden > 0 && (hidden * es) % 16 == 0,
                "trg_edge_anchor_loss: row width %d x %d bytes is not a multiple of 16 bytes", hidden, es);
  if ((int64_t)hidden * es > 1024) {   // checked here, not at dispatch, so n_rows = 0 is refused alike
    set_error("trg_edge_anchor_loss: rows wider than 1024 bytes are not supported (%d x %d bytes)", hidden, es);
    return TRG_E_UNSUPPORTED;
  }
  if (workspace == nullptr || workspace_bytes < trg_edge_bce_workspace_bytes(n_rows)) {
    set_error("trg_edge_anchor_loss: workspace %zu < required %zu", workspace_bytes,
              trg_edge_bce_workspace_bytes(n_rows));
    return TRG_E_WORKSPACE;
  }
  BceArgs a{};
  a.rowptr = rowptr; a.col_p = col; a.eid = eid; a.neg_p = nullptr;
  a.u = anchor; a.p = gathered; a.wbar = wbar; a.c_pos = coef_out; a.c_neg = nullptr; a.g_u = g_anchor;
  a.partials = reinterpret_cast<double*>(workspace);
  a.n_users = n_rows;
  a.inv_e = n_edges_scale > 0 ? (float)(1.0 / (double)n_edges_scale) : 0.f;
  a.row_vecs = hidden * es / 16;
  a.label = label ? 1 : 0;
  a.accumulate = accumulate ? 1 : 0;
  a.relu_gate = relu_gate ? 1 : 0;
  int64_t n_blocks = 0;
  if (n_rows > 0 && a.row_vecs == 32 && !anchor_ring_off()) {      // 512-byte rows: cp.async ring form
    n_blocks = ceil_div<int64_t>(n_rows, (int64_t)(kThreads / 32) * 4);
    static SmemAttrState attr_f32, attr_bf16;
    if (dtype == TRG_F32) {
      TRG_CUDA(ensure_dyn_smem(edge_anchor_ring<float>, kRingBytes, attr_f32));
      edge_anchor_ring<float><<<(unsigned)n_blocks, kThreads, kRingBytes, st>>>(a);
    } else {
      TRG_CUDA(ensure_dyn_smem(edge_anchor_ring<__nv_bfloat16>, kRingBytes, attr_bf16));
      edge_anchor_ring<__nv_bfloat16><<<(unsigned)n_blocks, kThreads, kRingBytes, st>>>(a);
    }
    count_launch();
    TRG_LAUNCH_OK();
  } else if (n_rows > 0) {
    int rc = dtype == TRG_F32 ? launch_bce<float, false>(a, &n_blocks, st, false)
                              : launch_bce<__nv_bfloat16, false>(a, &n_blocks, st, false);
    if (rc) return rc;
    count_launch();
    TRG_LAUNCH_OK();
  }
  edge_bce_finish<<<1, 1024, 0, st>>>(a.partials, n_blocks, wbar, (double)n_edges_scale, loss_out);
  count_launch();
  TRG_LAUNCH_OK();
  return TRG_OK;
}
