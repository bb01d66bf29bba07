// Weighted segment gather-sum over a CSR (SpMM with dense feature rows), sm_100a.
//
// Forward of the SAGE / RSAGE mean aggregation the three shipped configs use
//   SAGEConv.message + PyG mean aggr   models/gcn_lib/sparse/torch_vertex.py:279-286
// (the per-edge lin_r GEMM is hoisted AFTER the aggregation, SURVEY.md App. B.4), its backward
// (same kernel on the by-source CSR) and the source-side pass of the GENConv backward.
// Deterministic: a row's entries are summed in CSR order by one lane group, no atomics.
//
// Replicated topologies: train.py batches B patients that all share ONE edge list
// (dataloader/multiloader.py:687-698).  With replicas = B the CSR describes a single graph and the
// kernel walks it once per row while streaming all B feature rows, so index traffic drops B-fold and
// every entry issues RB independent row loads (memory-level parallelism even for 1-entry rows).
//
// HBM-bound: algorithmic bytes = 4*C*rows*2 + 8*nnz.
//
// Also here, because they share the row / lane-group / replica-slice geometry and the helpers:
//   * the fast replicated epilogue's extras -- the row's own src rows copied alongside (self_out: left half of cat(x, agg)),
//     addend, activation-derivative mask, fused output activation (mlg_gather_sum_act: transform-first SAGE layer);
//   * the backward of the fully factored first SAGE layer of MultilevelGNN: sage_rank1_bwd_rows_kernel
//     (mlg_sage_rank1_bwd_rows, by target row; its forward is in sage_rank1.cu).
#include <cstdlib>

#include "common.cuh"
#include "../../include/mlg_b200.h"

namespace {

constexpr int kThreads = 256;
#ifndef MLG_GS_UN
#define MLG_GS_UN 4
#endif
constexpr int UN = MLG_GS_UN;   // entries in flight (single-graph path)
#ifndef MLG_GS_RB
#define MLG_GS_RB 4
#endif
// min resident blocks per SM for the replicated kernel.  With plain __launch_bounds__(256) ptxas minimised registers by
// re-using ONE pair of float4 registers for all RB row loads of an entry, which serialised them into RB/2 dependent
// round trips (ncu source page: all stall samples on the first FFMA after each load pair).  RB = 4 with an explicit
// 3-blocks/SM budget (80 registers) makes it batch the four loads: 139 -> 102 us per SAGE aggregation at the gbm shape
// (RB = 8 / 2 blocks: 111 us, RB = 16 / 1 block: 129 us, RB = 2: 132 us).
#ifndef MLG_GS_MINB
#define MLG_GS_MINB 3
#endif
constexpr int RB = MLG_GS_RB;   // replicas in flight (replicated path)
// CSR entries per step of the replicated kernel (per-replica source rows): JU entries' rows (JU x RB loads per lane) are
// requested before the first FMA.  Measured at the gbm shape (one box, A/B libraries): JU = 2 (79 registers) 61.7 us vs 61.2 us
// for JU = 1, step 0.829 ms either way; JU = 4 (121 registers, 2 blocks/SM) 70.4 us, step 0.850 ms -- the kernel is not
// bound by the per-row chain of round trips, so the default stays 1.
#ifndef MLG_GS_JU
#define MLG_GS_JU 1
#endif
constexpr int JUX = MLG_GS_JU;

struct GsP {
  const float* src;
  const int* rowptr;
  const int* idx;
  const float* val;
  const float* pre;
  const float* post;
  const float* addend;
  const float* red_scale;   // optional [replicas*n]: out[slice*n + row] = sum_{b in slice} red_scale[b*n+row] * result_b (replicated path)
  const float* mask;     // optional: out *= (mask[row, c] > 0 ? 1 : mask_slope)  (activation derivative of the consumer's input)
  const int* order;      // optional row visiting order (heavy rows first, equal degrees together)
  float* out;
  float* self_out;
  unsigned ld_src, ld_out, ld_add, ld_self, ld_mask;
  float mask_slope;
  int n, C, post_mode, relative;
  int replicas;
  unsigned rep_rows_src;   // 0: every replica reads the SAME src rows (rank-1 source, pre is per replica)
  unsigned rep_rows_pre;   // rows per replica of `pre` (0: shared)
  float act_slope;
  int act;                 // fast replicated epilogue: out = LeakyReLU_act_slope(out) after addend / mask
};

__device__ __forceinline__ const float* rowp(const float* b, unsigned r, unsigned ld) { return b + (size_t)r * ld; }
__device__ __forceinline__ float* rowp(float* b, unsigned r, unsigned ld) { return b + (size_t)r * ld; }

template <int VEC>
__device__ __forceinline__ void ldv(float (&d)[VEC], const float* p, bool ok) {
  if (VEC == 4) {
    const float4 t = ok ? ld_gather4(p) : make_float4(0.f, 0.f, 0.f, 0.f);
    d[0] = t.x; d[1 % VEC] = t.y; d[2 % VEC] = t.z; d[3 % VEC] = t.w;
  } else {
    d[0] = ok ? __ldg(p) : 0.f;
  }
}
// unconditional load that cannot be sunk below later arithmetic
// (measured: the same load with L1::no_allocate -- the gathered rows are not re-used by this SM -- is SLOWER, 72 -> 94 us per
// launch at the gbm shape; the plain read-only path it is)
template <int VEC>
__device__ __forceinline__ void ldv_now(float (&d)[VEC], const float* p) {
  if (VEC == 4) {
    asm volatile("ld.global.nc.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(d[0]), "=f"(d[1 % VEC]), "=f"(d[2 % VEC]), "=f"(d[3 % VEC])
                 : "l"(p));
  } else {
    asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(d[0]) : "l"(p));
  }
}
template <int VEC>
__device__ __forceinline__ void stv(float* p, const float (&d)[VEC], bool ok) {
  if (!ok) return;
  if (VEC == 4) st4(p, make_float4(d[0], d[1 % VEC], d[2 % VEC], d[3 % VEC]));
  else p[0] = d[0];
}

// finish one output row: post scale, relative term, addend, stores
template <int VEC>
__device__ __forceinline__ void finish_row(const GsP& P, float (&acc)[VEC], unsigned out_row, unsigned src_row,
                                           unsigned c, bool cok, float postf, int cnt_row, float self_scale = 1.f) {
#pragma unroll
  for (int k = 0; k < VEC; ++k) acc[k] *= postf;
  if (P.relative || P.self_out) {
    float xs[VEC];
    ldv<VEC>(xs, rowp(P.src, src_row, P.ld_src) + c, cok);
#pragma unroll
    for (int k = 0; k < VEC; ++k) xs[k] *= self_scale;
    if (P.relative) {
      const float f = (P.post_mode == 1) ? (cnt_row > 0 ? 1.f : 0.f) : (float)cnt_row * postf;
#pragma unroll
      for (int k = 0; k < VEC; ++k) acc[k] -= f * xs[k];
    }
    if (P.self_out) stv<VEC>(rowp(P.self_out, out_row, P.ld_self) + c, xs, cok);
  }
  if (P.addend) {
    float ad[VEC];
    ldv<VEC>(ad, rowp(P.addend, out_row, P.ld_add) + c, cok);
#pragma unroll
    for (int k = 0; k < VEC; ++k) acc[k] += ad[k];
  }
  if (P.mask) {
    float mk[VEC];
    ldv<VEC>(mk, rowp(P.mask, out_row, P.ld_mask) + c, cok);
#pragma unroll
    for (int k = 0; k < VEC; ++k) acc[k] *= mk[k] > 0.f ? 1.f : P.mask_slope;
  }
  stv<VEC>(rowp(P.out, out_row, P.ld_out) + c, acc, cok);
}

// ---------------------------------------------------------------------------------------------
// single-graph path: one lane group per row, UN entries in flight
// ---------------------------------------------------------------------------------------------
// Rows longer than kHeavy entries (hubs: the by-source CSR of a kNN graph has out-degrees in the thousands while the
// mean is k) are NOT walked by their one lane group -- a single group with UN loads in flight would be the kernel's
// tail (measured: 610 us for an 820 MB gather at N=100k, k=16, H=128, max out-degree 1502).  The group only records the
// row; after the block's light rows are done ALL lane groups of the block walk each recorded row together (group g takes
// entry blocks g, g+G, ...), partial sums meet in shared memory and are added in group order: still a fixed summation
// order, no atomics on the data.
constexpr int kHeavy = 96;

template <int LANES, int VEC>
__device__ __forceinline__ void gs_accumulate(const GsP& P, const float* sc, bool cok, unsigned gmask, int sl, int first,
                                              int end, int stride, float (&acc)[VEC]) {
  for (int base = first; base < end; base += stride) {
    const int q = min(base + sl, end - 1);
    const unsigned my_idx = (unsigned)__ldg(P.idx + q);
    float my_w = P.val ? __ldg(P.val + q) : 1.f;
    if (P.pre) my_w *= __ldg(P.pre + my_idx);
    const int cnt = min(LANES, end - base);
    for (int j = 0; j < cnt; j += UN) {
      float xv[UN][VEC];
      float w[UN];
#pragma unroll
      for (int u = 0; u < UN; ++u) {
        const int jj = min(j + u, cnt - 1);
        const unsigned s = __shfl_sync(gmask, my_idx, jj, LANES);
        w[u] = __shfl_sync(gmask, my_w, jj, LANES);
        if (j + u >= cnt) w[u] = 0.f;
        ldv<VEC>(xv[u], rowp(sc, s, P.ld_src), cok);
      }
#pragma unroll
      for (int u = 0; u < UN; ++u)
#pragma unroll
        for (int k = 0; k < VEC; ++k) acc[k] = fmaf(w[u], xv[u][k], acc[k]);
    }
  }
}

template <int LANES, int VEC>
__global__ void __launch_bounds__(kThreads) gather_sum_kernel(const GsP P) {
  constexpr int RPW = 32 / LANES;
  constexpr int CW = LANES * VEC;
  constexpr int G = kThreads / LANES;          // lane groups per block
  __shared__ int heavy_rows[G];
  __shared__ int n_heavy;
  __shared__ float part[G * CW];
  const int lane = threadIdx.x & 31;
  const int sub = lane / LANES, sl = lane % LANES;
  const unsigned gmask = (LANES == 32) ? 0xffffffffu : (((1u << LANES) - 1u) << (sub * LANES));
  const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long slot = warp * RPW + sub;
  const int C = P.C;
  const int nchunks = (C + CW - 1) / CW;
  if (threadIdx.x == 0) n_heavy = 0;
  __syncthreads();
  if (slot < P.n) {
    const long long row = P.order ? __ldg(P.order + slot) : slot;
    const int beg = __ldg(P.rowptr + row), end = __ldg(P.rowptr + row + 1);
    const int cnt_row = end - beg;
    if (cnt_row > kHeavy) {
      if (sl == 0) heavy_rows[atomicAdd(&n_heavy, 1)] = (int)row;   // list order is irrelevant: rows are independent
    } else {
      float postf = 1.f;
      if (P.post_mode == 1) postf = cnt_row > 0 ? 1.f / (float)cnt_row : 0.f;
      else if (P.post_mode == 2) postf = __ldg(P.post + row);
      for (int ch = 0; ch < nchunks; ++ch) {
        const unsigned c = ch * CW + sl * VEC;
        const bool cok = c < (unsigned)C;
        float acc[VEC];
#pragma unroll
        for (int k = 0; k < VEC; ++k) acc[k] = 0.f;
        gs_accumulate<LANES, VEC>(P, P.src + c, cok, gmask, sl, beg, end, LANES, acc);
        finish_row<VEC>(P, acc, (unsigned)row, (unsigned)row, c, cok, postf, cnt_row);
      }
    }
  }
  __syncthreads();
  const int nh = n_heavy;
  if (nh == 0) return;
  const int g = threadIdx.x / LANES;
  for (int h = 0; h < nh; ++h) {
    const int row = heavy_rows[h];
    const int beg = __ldg(P.rowptr + row), end = __ldg(P.rowptr + row + 1);
    const int cnt_row = end - beg;
    float postf = 1.f;
    if (P.post_mode == 1) postf = 1.f / (float)cnt_row;
    else if (P.post_mode == 2) postf = __ldg(P.post + row);
    for (int ch = 0; ch < nchunks; ++ch) {
      const unsigned c = ch * CW + sl * VEC;
      const bool cok = c < (unsigned)C;
      float acc[VEC];
#pragma unroll
      for (int k = 0; k < VEC; ++k) acc[k] = 0.f;
      gs_accumulate<LANES, VEC>(P, P.src + c, cok, gmask, sl, beg + g * LANES, end, G * LANES, acc);
#pragma unroll
      for (int k = 0; k < VEC; ++k) part[g * CW + sl * VEC + k] = acc[k];
      __syncthreads();
      if (g == 0) {
#pragma unroll 4
        for (int gg = 1; gg < G; ++gg)
#pragma unroll
          for (int k = 0; k < VEC; ++k) acc[k] += part[gg * CW + sl * VEC + k];
        finish_row<VEC>(P, acc, (unsigned)row, (unsigned)row, c, cok, postf, cnt_row);
      }
      __syncthreads();
    }
  }
}

// ---------------------------------------------------------------------------------------------
// replicated path: the CSR covers ONE graph (n rows); replica b reads src rows b*rep_rows_src + idx and
// writes out rows b*n + row.  RB replicas are accumulated at once.
// RANK1: every replica reads the SAME src rows and differs only by the per-(replica,row) scalar `pre`
//        (MultilevelGNN layer 0: x0[b,n,:] = x[b,n] * node_embedding[n,:] is never materialised).
// ---------------------------------------------------------------------------------------------
template <int LANES, int VEC, bool RANK1, bool RED = false>
__global__ void __launch_bounds__(kThreads, MLG_GS_MINB) gather_sum_rep_kernel(const GsP P, int gy) {
  constexpr int RPW = 32 / LANES;
  constexpr int CW = LANES * VEC;
  constexpr int JU = RANK1 ? 2 : JUX;   // entries per step
  const int lane = threadIdx.x & 31;
  const int sub = lane / LANES, sl = lane % LANES;
  const unsigned gmask = (LANES == 32) ? 0xffffffffu : (((1u << LANES) - 1u) << (sub * LANES));
  // 1-D grid, replica slice fastest: heavy rows (order[] is sorted by degree) of ALL slices start first
  // (slice-slowest, i.e. a 4x smaller live working set in L2, measured SLOWER: 161 vs 139 us at the gbm shape)
  const int ychunk = blockIdx.x % gy;
  const long long rowblock = blockIdx.x / gy;
  const long long warp = (rowblock * (long long)blockDim.x + threadIdx.x) >> 5;
  const int rep_per_y = (P.replicas + gy - 1) / gy;
  const int b_lo = ychunk * rep_per_y, b_hi = min(P.replicas, b_lo + rep_per_y);
  const long long slot = warp * RPW + sub;
  if (slot >= P.n || b_lo >= b_hi) return;
  const unsigned row = P.order ? (unsigned)__ldg(P.order + slot) : (unsigned)slot;
  const int C = P.C;
  const int beg = __ldg(P.rowptr + row), end = __ldg(P.rowptr + row + 1);
  const int cnt_row = end - beg;
  float postf = 1.f;
  if (P.post_mode == 1) postf = cnt_row > 0 ? 1.f / (float)cnt_row : 0.f;
  else if (P.post_mode == 2) postf = __ldg(P.post + row);
  const bool shared_pre = P.pre != nullptr && P.rep_rows_pre == 0;
  // first LANES entries of the row live in registers for the whole replica loop
  unsigned idx0 = 0;
  float w0 = 0.f;
  if (cnt_row > 0) {
    const int q = min(beg + sl, end - 1);
    idx0 = (unsigned)__ldg(P.idx + q);
    w0 = P.val ? __ldg(P.val + q) : 1.f;
    if (shared_pre) w0 *= __ldg(P.pre + idx0);
  }
  const int nchunks = (C + CW - 1) / CW;
  for (int ch = 0; ch < nchunks; ++ch) {
    const unsigned c = ch * CW + sl * VEC;
    const bool cok = c < (unsigned)C;
    const float* sc = P.src + (cok ? c : 0u);   // lanes past C read (and discard) the row start: no predicated loads
    const size_t rep_stride = (size_t)P.rep_rows_src * P.ld_src;
    float red[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) red[k] = 0.f;
    for (int b0 = b_lo; b0 < b_hi; b0 += RB) {
      const int nb = min(RB, b_hi - b0);
      float acc[RB][VEC];
#pragma unroll
      for (int r = 0; r < RB; ++r)
#pragma unroll
        for (int k = 0; k < VEC; ++k) acc[r][k] = 0.f;
      for (int base = beg; base < end; base += LANES) {
        unsigned my_idx = idx0;
        float my_w = w0;
        if (base != beg) {
          const int q = min(base + sl, end - 1);
          my_idx = (unsigned)__ldg(P.idx + q);
          my_w = P.val ? __ldg(P.val + q) : 1.f;
          if (shared_pre) my_w *= __ldg(P.pre + my_idx);
        }
        const int cnt = min(LANES, end - base);
        for (int j = 0; j < cnt; j += JU) {
          if (RANK1) {
            unsigned s[JU];
            float w[JU], xv[JU][VEC], pw[JU][RB];
#pragma unroll
            for (int u = 0; u < JU; ++u) {
              const int jj = min(j + u, cnt - 1);
              s[u] = __shfl_sync(gmask, my_idx, jj, LANES);
              w[u] = __shfl_sync(gmask, my_w, jj, LANES);
              if (j + u >= cnt) w[u] = 0.f;
              ldv<VEC>(xv[u], rowp(sc, s[u], P.ld_src), cok);
#pragma unroll
              for (int r = 0; r < RB; ++r) {
                const int b = min(b0 + r, b_hi - 1);
                pw[u][r] = __ldg(P.pre + (size_t)b * P.rep_rows_pre + s[u]);
              }
            }
#pragma unroll
            for (int u = 0; u < JU; ++u)
#pragma unroll
              for (int r = 0; r < RB; ++r) {
                const float f = w[u] * pw[u][r];
#pragma unroll
                for (int k = 0; k < VEC; ++k) acc[r][k] = fmaf(f, xv[u][k], acc[r][k]);
              }
          } else {
            unsigned s[JU];
            float w[JU], xv[JU][RB][VEC];
#pragma unroll
            for (int u = 0; u < JU; ++u) {
              const int jj = min(j + u, cnt - 1);     // past the end: re-request the last entry's rows (L1 hits), not added
              s[u] = __shfl_sync(gmask, my_idx, jj, LANES);
              w[u] = __shfl_sync(gmask, my_w, jj, LANES);
            }
            // all JU * RB row loads are issued before the first FMA (volatile asm keeps ptxas from re-using one pair of
            // registers for the loads, which serialised them into RB/2 round trips: ncu source page, r01)
#pragma unroll
            for (int u = 0; u < JU; ++u) {
              const float* p0 = rowp(sc, (unsigned)b0 * P.rep_rows_src + s[u], P.ld_src);
#pragma unroll
              for (int r = 0; r < RB; ++r) ldv_now<VEC>(xv[u][r], p0 + (size_t)min(r, nb - 1) * rep_stride);
            }
#pragma unroll
            for (int u = 0; u < JU; ++u)      // entries in CSR order: the same sequence of FMAs for every JU
              if (u == 0 || j + u < cnt) {
#pragma unroll
                for (int r = 0; r < RB; ++r)
#pragma unroll
                  for (int k = 0; k < VEC; ++k) acc[r][k] = fmaf(w[u], xv[u][r][k], acc[r][k]);
              }
          }
        }
      }
      if (!RANK1 && !P.relative) {
        // backward-style epilogue (addend / activation mask): request ALL replicas' addend and mask rows first, then
        // finish -- one exposed load latency per thread instead of RB sequential ones (the masked backward aggregation
        // ran 180 us against 138 us unmasked with the row-by-row epilogue)
        // (two phases -- addend rows, then mask rows -- so that only RB rows are live next to the accumulators)
        float t[RB][VEC];
        if (P.self_out) {   // left half of cat(x, agg): the row's own src rows, copied with batched loads
#pragma unroll
          for (int r = 0; r < RB; ++r)
            ldv<VEC>(t[r], rowp(P.src, (unsigned)min(b0 + r, b_hi - 1) * P.rep_rows_src + row, P.ld_src) + c, cok);
#pragma unroll
          for (int r = 0; r < RB; ++r)
            if (b0 + r < b_hi) stv<VEC>(rowp(P.self_out, (unsigned)(b0 + r) * (unsigned)P.n + row, P.ld_self) + c, t[r], cok);
        }
        if (P.addend) {
#pragma unroll
          for (int r = 0; r < RB; ++r)
            ldv<VEC>(t[r], rowp(P.addend, (unsigned)min(b0 + r, b_hi - 1) * (unsigned)P.n + row, P.ld_add) + c, cok);
#pragma unroll
          for (int r = 0; r < RB; ++r)
#pragma unroll
            for (int k = 0; k < VEC; ++k) acc[r][k] = fmaf(acc[r][k], postf, t[r][k]);
        } else {
#pragma unroll
          for (int r = 0; r < RB; ++r)
#pragma unroll
            for (int k = 0; k < VEC; ++k) acc[r][k] *= postf;
        }
        if (P.mask) {
#pragma unroll
          for (int r = 0; r < RB; ++r)
            ldv<VEC>(t[r], rowp(P.mask, (unsigned)min(b0 + r, b_hi - 1) * (unsigned)P.n + row, P.ld_mask) + c, cok);
#pragma unroll
          for (int r = 0; r < RB; ++r)
#pragma unroll
            for (int k = 0; k < VEC; ++k) acc[r][k] *= t[r][k] > 0.f ? 1.f : P.mask_slope;
        }
        if (P.act) {
#pragma unroll
          for (int r = 0; r < RB; ++r)
#pragma unroll
            for (int k = 0; k < VEC; ++k) acc[r][k] = acc[r][k] > 0.f ? acc[r][k] : acc[r][k] * P.act_slope;
        }
        if (RED) {   // weighted reduction over the replicas instead of one output row per replica
#pragma unroll
          for (int r = 0; r < RB; ++r) {
            const float w = (b0 + r < b_hi) ? __ldg(P.red_scale + (size_t)(b0 + r) * P.n + row) : 0.f;
#pragma unroll
            for (int k = 0; k < VEC; ++k) red[k] = fmaf(w, acc[r][k], red[k]);
          }
        } else {
#pragma unroll
          for (int r = 0; r < RB; ++r)
            if (b0 + r < b_hi) stv<VEC>(rowp(P.out, (unsigned)(b0 + r) * (unsigned)P.n + row, P.ld_out) + c, acc[r], cok);
        }
      } else if (RANK1 && !P.relative && !P.addend && !P.mask && P.self_out) {
        // first-layer epilogue: the self row (one embedding row for ALL replicas) and the RB per-replica scalars are
        // requested together; then 2*RB stores
        float es[VEC], sc[RB];
        ldv<VEC>(es, rowp(P.src, row, P.ld_src) + c, cok);
#pragma unroll
        for (int r = 0; r < RB; ++r) sc[r] = __ldg(P.pre + (size_t)min(b0 + r, b_hi - 1) * P.rep_rows_pre + row);
#pragma unroll
        for (int r = 0; r < RB; ++r) {
          if (b0 + r < b_hi) {
            const unsigned orow = (unsigned)(b0 + r) * (unsigned)P.n + row;
            float xs[VEC];
#pragma unroll
            for (int k = 0; k < VEC; ++k) {
              xs[k] = es[k] * sc[r];
              acc[r][k] *= postf;
            }
            stv<VEC>(rowp(P.self_out, orow, P.ld_self) + c, xs, cok);
            stv<VEC>(rowp(P.out, orow, P.ld_out) + c, acc[r], cok);
          }
        }
      } else {
#pragma unroll
        for (int r = 0; r < RB; ++r) {
          const int b = b0 + r;
          if (b < b_hi) {
            const float self_scale = RANK1 ? __ldg(P.pre + (size_t)b * P.rep_rows_pre + row) : 1.f;
            finish_row<VEC>(P, acc[r], (unsigned)b * (unsigned)P.n + row, (unsigned)b * P.rep_rows_src + row, c, cok,
                            postf, cnt_row, self_scale);
          }
        }
      }
    }
    if (RED) stv<VEC>(rowp(P.out, (unsigned)ychunk * (unsigned)P.n + row, P.ld_out) + c, red, cok);
  }
}

// ---------------------------------------------------------------------------------------------
// Fully factored first SAGE layer, backward w.r.t. the tables (mlg_sage_rank1_bwd_rows), organised by TARGET row so
// that gz is read exactly once:
// one warp per row i; lane l owns channels l, l+32, ... and keeps gz[b,i,channel] of 32 replicas in registers
// (coalesced 128-byte loads, all in flight together); then for every entry q of the row (source j)
//     h[q,:] = (val_q / cnt_i) * sum_b x[b,j] gz[b,i,:]
// -- a 32-term dot per channel with x[.,j] broadcast by shuffles -- plus the two per-row reductions
//     g_self[i,:] = sum_b x[b,i] gz[b,i,:]        g_bias_rows[i,:] = sum_b gz[b,i,:].
// g_E_nbr[j,:] = sum_{q: idx_q = j} h[q,:] is then a segment sum over the by-source CSR (mlg_gather_sum, single graph):
// fixed order, no atomics.  More than 32 replicas: further passes accumulate into the same outputs.
// ---------------------------------------------------------------------------------------------
struct R1B {
  const float* gz;
  const unsigned long long* mbits;   // optional (C == 64): sign bits of y written by sage_rank1_fwd_rows_kernel, [n][B]
  const float* y;      // optional: gz is dL/dy of this layer's LeakyReLU output y; the kernel applies the derivative
  float slope;
  const float* xs;
  const int* rowptr;
  const int* idx;
  const float* val;
  const int* order;
  float* h;
  float* g_self;
  float* g_bias_rows;
  unsigned ld_g, ld_self;
  int n, B;
  int xs_t;            // xs is the transposed node-value matrix [n][B] (one coalesced load per entry) instead of [B][n]
  int gz_nm;           // gz (and y) rows node-major: (replica b, node i) at i * B + b instead of b * n + i
};

#ifndef MLG_R1B_MINB
#define MLG_R1B_MINB 2     // resident blocks per SM (register budget 128; 1 -> 255)
#endif
#ifndef MLG_R1B_YB
#define MLG_R1B_YB 8       // replicas whose y values (self-masking) are requested together
#endif

// PACKED (C == 64, B % 32 == 0, transposed node values): the per-entry dot products over the 32 replicas run on replica
// PAIRS -- the gradient rows are packed once per gene, the neighbour's replica values come back from a warp-private
// shared-memory row as eight broadcast LDS.128 (16 register pairs), so an entry costs 8 LDS.128 + 32 FFMA2 instead of
// 32 SHFL + 64 FFMA (same restructuring as sage_rank1.cu's forward; the even / odd replica halves are added at the end).
template <int CPL, bool PACKED>
__global__ void __launch_bounds__(kThreads, MLG_R1B_MINB) sage_rank1_bwd_rows_kernel(const R1B P) {
  constexpr int C = 32 * CPL;
  constexpr int EU = 4;   // entries whose x loads are in flight together
  __shared__ __align__(16) float xsm_all[PACKED ? kThreads / 32 : 1][EU][32];
  float* xsm = &xsm_all[PACKED ? (threadIdx.x >> 5) : 0][0][0];
  const int lane = threadIdx.x & 31;
  const long long slot = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (slot >= P.n) return;
  const unsigned row = P.order ? (unsigned)__ldg(P.order + slot) : (unsigned)slot;
  const int beg = __ldg(P.rowptr + row), end = __ldg(P.rowptr + row + 1);
  const float inv = end > beg ? 1.f / (float)(end - beg) : 0.f;
  for (int rb0 = 0; rb0 < P.B; rb0 += 32) {
    const int nb = min(32, P.B - rb0);
    const bool first = rb0 == 0;
    float g[CPL][32];
    const size_t rstride = P.gz_nm ? (size_t)P.ld_g : (size_t)P.n * P.ld_g;      // replica to replica
    const size_t rbase = (P.gz_nm ? (size_t)row * P.B + rb0 : (size_t)rb0 * P.n + row) * P.ld_g + lane;
    const float* gp = P.gz + rbase;
#pragma unroll
    for (int b = 0; b < 32; ++b)
#pragma unroll
      for (int k = 0; k < CPL; ++k) g[k][b] = b < nb ? __ldg(gp + (size_t)b * rstride + 32 * k) : 0.f;
    if (P.mbits) {   // gz arrived as dL/dy: LeakyReLU'(y) from the forward kernel's sign bits (one 8-byte word per replica)
      const unsigned long long wd = lane < nb ? __ldg(P.mbits + (size_t)row * P.B + rb0 + lane) : ~0ull;
      const unsigned lo = (unsigned)wd, hi = (unsigned)(wd >> 32);
      const int pos = (lane & 3) * 16 + (lane >> 2);    // channel `lane`; channel lane + 32 sits 8 bits higher
#pragma unroll
      for (int b = 0; b < 32; ++b) {
        const unsigned long long w =
            ((unsigned long long)__shfl_sync(0xffffffffu, hi, b) << 32) | __shfl_sync(0xffffffffu, lo, b);
        g[0][b] *= ((w >> pos) & 1ull) ? 1.f : P.slope;
        if (CPL == 2) g[CPL - 1][b] *= ((w >> (pos + 8)) & 1ull) ? 1.f : P.slope;
      }
    } else if (P.y) {   // gz arrived as dL/dy: multiply by LeakyReLU'(y) (y has the layout of gz); 8 replicas' y values at a time
      const float* yp = P.y + rbase;
#pragma unroll
      for (int b8 = 0; b8 < 32; b8 += MLG_R1B_YB) {
        float yv[CPL][MLG_R1B_YB];
#pragma unroll
        for (int b = 0; b < MLG_R1B_YB; ++b)
#pragma unroll
          for (int k = 0; k < CPL; ++k) yv[k][b] = b8 + b < nb ? __ldg(yp + (size_t)(b8 + b) * rstride + 32 * k) : 1.f;
#pragma unroll
        for (int b = 0; b < MLG_R1B_YB; ++b)
#pragma unroll
          for (int k = 0; k < CPL; ++k) g[k][b8 + b] *= yv[k][b] > 0.f ? 1.f : P.slope;
      }
    }
    // lane b reads replica rb0+b (clamped; masked below): element (replica, node) = xp[node * xstride]
    const float* xp = P.xs_t ? P.xs + rb0 + min(lane, nb - 1) : P.xs + (size_t)(rb0 + min(lane, nb - 1)) * P.n;
    const size_t xstride = P.xs_t ? (size_t)P.B : 1;
    const float lane_live = lane < nb ? 1.f : 0.f;
    u64 gp2[PACKED ? CPL : 1][PACKED ? 16 : 1];   // (replica 2j, replica 2j + 1) of this lane's channels
    if constexpr (PACKED) {
#pragma unroll
      for (int k = 0; k < CPL; ++k)
#pragma unroll
        for (int j = 0; j < 16; ++j) gp2[k][j] = pk2(g[k][2 * j], g[k][2 * j + 1]);
    }
    {
      const float xv = __ldg(xp + row * xstride) * lane_live;
      float e1[CPL], gb[CPL];
      if constexpr (PACKED) {
        xsm[lane] = xv;
        __syncwarp();
        u64 e2[CPL], b2[CPL];
#pragma unroll
        for (int k = 0; k < CPL; ++k) e2[k] = b2[k] = 0ull;
        const ulonglong2* xq = reinterpret_cast<const ulonglong2*>(xsm);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const ulonglong2 v = xq[i];
#pragma unroll
          for (int k = 0; k < CPL; ++k) {
            e2[k] = fma2(v.x, gp2[k][2 * i], e2[k]);
            e2[k] = fma2(v.y, gp2[k][2 * i + 1], e2[k]);
            b2[k] = add2(b2[k], gp2[k][2 * i]);
            b2[k] = add2(b2[k], gp2[k][2 * i + 1]);
          }
        }
#pragma unroll
        for (int k = 0; k < CPL; ++k) {
          float lo, hi;
          upk2(e2[k], lo, hi);
          e1[k] = lo + hi;
          upk2(b2[k], lo, hi);
          gb[k] = lo + hi;
        }
        __syncwarp();
      } else {
#pragma unroll
        for (int k = 0; k < CPL; ++k) e1[k] = gb[k] = 0.f;
#pragma unroll
        for (int b = 0; b < 32; ++b) {
          const float xb = __shfl_sync(0xffffffffu, xv, b);
#pragma unroll
          for (int k = 0; k < CPL; ++k) {
            e1[k] = fmaf(xb, g[k][b], e1[k]);
            gb[k] += g[k][b];
          }
        }
      }
#pragma unroll
      for (int k = 0; k < CPL; ++k) {
        float* ps = P.g_self + (size_t)row * P.ld_self + lane + 32 * k;
        float* pb = P.g_bias_rows + (size_t)row * C + lane + 32 * k;
        *ps = first ? e1[k] : *ps + e1[k];
        *pb = first ? gb[k] : *pb + gb[k];
      }
    }
    for (int base = beg; base < end; base += 32) {
      const int q = min(base + lane, end - 1);
      const unsigned my_idx = (unsigned)__ldg(P.idx + q);
      const float my_w = (P.val ? __ldg(P.val + q) : 1.f) * inv;
      const int cnt = min(32, end - base);
      for (int j = 0; j < cnt; j += EU) {
        float xv[EU];
#pragma unroll
        for (int u = 0; u < EU; ++u) {
          const unsigned s = __shfl_sync(0xffffffffu, my_idx, min(j + u, cnt - 1));
          xv[u] = __ldg(xp + s * xstride) * lane_live;
        }
        if constexpr (PACKED) {
#pragma unroll
          for (int u = 0; u < EU; ++u) xsm[u * 32 + lane] = xv[u];
          __syncwarp();
        }
#pragma unroll
        for (int u = 0; u < EU; ++u) {
          if (j + u < cnt) {   // warp-uniform
            const float w = __shfl_sync(0xffffffffu, my_w, j + u);
            float hk[CPL];
            if constexpr (PACKED) {
              u64 h2[CPL];
#pragma unroll
              for (int k = 0; k < CPL; ++k) h2[k] = 0ull;
              const ulonglong2* xq = reinterpret_cast<const ulonglong2*>(xsm + u * 32);
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const ulonglong2 v = xq[i];
#pragma unroll
                for (int k = 0; k < CPL; ++k) {
                  h2[k] = fma2(v.x, gp2[k][2 * i], h2[k]);
                  h2[k] = fma2(v.y, gp2[k][2 * i + 1], h2[k]);
                }
              }
#pragma unroll
              for (int k = 0; k < CPL; ++k) {
                float lo, hi;
                upk2(h2[k], lo, hi);
                hk[k] = lo + hi;
              }
            } else {
#pragma unroll
              for (int k = 0; k < CPL; ++k) hk[k] = 0.f;
#pragma unroll
              for (int b = 0; b < 32; ++b) {
                const float xb = __shfl_sync(0xffffffffu, xv[u], b);
#pragma unroll
                for (int k = 0; k < CPL; ++k) hk[k] = fmaf(xb, g[k][b], hk[k]);
              }
            }
#pragma unroll
            for (int k = 0; k < CPL; ++k) {
              float* ph = P.h + (size_t)(base + j + u) * C + lane + 32 * k;
              *ph = first ? w * hk[k] : fmaf(w, hk[k], *ph);
            }
          }
        }
        if constexpr (PACKED) __syncwarp();   // the next batch overwrites the rows
      }
    }
  }
}

// Negative result kept for the record (r01): a shared-memory staged variant of the replicated path (16-byte cp.async
// per lane into a per-warp ring, 12-16 entries in flight, the layout gen_aggr.cu's ring kernel uses) ran at
// 221-293 us against 134 us for the register-staged kernel above on the gbm shape: cp.async gathers top out near
// 4-4.5 TB/s on this part, below what plain LDG.128 gathers served from L2 reach (6.5-8.6 TB/s).  What did help was
// getting ptxas to issue all RB row loads before the first FMA (see MLG_GS_MINB).

// ---------------------------------------------------------------------------------------------
// Replicated aggregation over a NODE-MAJOR source (C == 32): src row of (replica b, node j) is j * B + b, so the B replica
// rows a CSR entry gathers are ONE contiguous 128 * B-byte block instead of B rows 128 * n * ld bytes apart.  A warp owns one
// output row for 16 replicas: lane (q, sl) = (lane / 8, lane % 8) covers bytes 16 * sl of replica 4 j + q, so every load
// instruction of the warp reads 512 contiguous bytes and an entry's four loads 2 KB (gather_sum_rep_kernel<8, 4>: four
// 128-byte rows of four unrelated nodes per instruction; the same bytes through L2, at a coarser request granularity).
// Both aggregations of the transform-first SAGE layer run here when the model hands it node-major rows: forward on the V half
// of the node-major [U | V] GEMM output (addend U, mean, LeakyReLU; its OUTPUT graph-major for the pool and the caller),
// backward on the gradient the pool backward writes node-major (mlg_pool_bwd_layout), out / self_out = [g_U | g_V] in the row
// order of the layer's input.
// ---------------------------------------------------------------------------------------------
constexpr int NM_JU = 2;   // CSR entries in flight per lane (8 row loads)
struct NmP {
  const float* src;      // node-major rows of 32 floats, leading dimension ld_src
  const int* rowptr;
  const int* idx;
  const float* val;
  const float* pre;      // optional [n]: weight *= pre[idx]
  const int* order;
  const float* addend;   // optional node-major rows (leading dimension ld_add): out = addend + post * sum
  float* out;
  float* self_out;       // optional: the row's own src rows copied alongside
  unsigned ld_src, ld_add, ld_out, ld_self;
  int n, B;
  int mean;              // post = 1 / row length (0 for an empty row) instead of 1
  int act;               // LeakyReLU(act_slope) on the result
  float act_slope;
  int out_nm;            // out / self_out rows node-major as well (else graph-major: b * n + i)
};
__global__ void __launch_bounds__(kThreads, 3) gather_nm_kernel(const NmP P) {
  const int lane = threadIdx.x & 31;
  const int q = lane >> 3, sl = lane & 7;
  const int B = P.B, n = P.n;
  const int halves = (B + 15) / 16;
  const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long slot = wid / halves;
  if (slot >= n) return;
  const int b_base = (int)(wid % halves) * 16;
  const unsigned row = P.order ? (unsigned)__ldg(P.order + slot) : (unsigned)slot;
  const int beg = __ldg(P.rowptr + row), end = __ldg(P.rowptr + row + 1);
  int bq[4];          // this lane's replica per load, clamped for the loads (stores test the unclamped value)
#pragma unroll
  for (int j = 0; j < 4; ++j) bq[j] = min(b_base + 4 * j + q, B - 1);
  float acc[4][4];
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int k = 0; k < 4; ++k) acc[j][k] = 0.f;
  const float* sc = P.src + sl * 4;
  for (int base = beg; base < end; base += 32) {
    const int p = min(base + lane, end - 1);
    const unsigned my_idx = (unsigned)__ldg(P.idx + p);
    float my_w = P.val ? __ldg(P.val + p) : 1.f;
    if (P.pre) my_w *= __ldg(P.pre + my_idx);
    const int cnt = min(32, end - base);
    for (int e = 0; e < cnt; e += NM_JU) {
      float4 v[NM_JU][4];
      float w[NM_JU];
#pragma unroll
      for (int u = 0; u < NM_JU; ++u) {
        const int ee = min(e + u, cnt - 1);
        const unsigned s = __shfl_sync(0xffffffffu, my_idx, ee);
        w[u] = (e + u < cnt) ? __shfl_sync(0xffffffffu, my_w, ee) : 0.f;
        const float* ps = sc + (size_t)s * B * P.ld_src;
#pragma unroll
        for (int j = 0; j < 4; ++j) v[u][j] = ld_gather4(ps + (size_t)bq[j] * P.ld_src);
      }
#pragma unroll
      for (int u = 0; u < NM_JU; ++u)      // entries in CSR order: one fixed sequence of FMAs per output element
        if (u == 0 || e + u < cnt) {       // (a padded entry is not added: -0.0 / NaN safe, and the sequence gather_sum_rep runs)
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            acc[j][0] = fmaf(w[u], v[u][j].x, acc[j][0]);
            acc[j][1] = fmaf(w[u], v[u][j].y, acc[j][1]);
            acc[j][2] = fmaf(w[u], v[u][j].z, acc[j][2]);
            acc[j][3] = fmaf(w[u], v[u][j].w, acc[j][3]);
          }
        }
    }
  }
  const float postf = P.mean ? (end > beg ? 1.f / (float)(end - beg) : 0.f) : 1.f;
  float4 t[4];
  if (P.addend) {
#pragma unroll
    for (int j = 0; j < 4; ++j) t[j] = ld_gather4(P.addend + ((size_t)row * B + bq[j]) * P.ld_add + sl * 4);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      acc[j][0] = fmaf(acc[j][0], postf, t[j].x);
      acc[j][1] = fmaf(acc[j][1], postf, t[j].y);
      acc[j][2] = fmaf(acc[j][2], postf, t[j].z);
      acc[j][3] = fmaf(acc[j][3], postf, t[j].w);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int k = 0; k < 4; ++k) acc[j][k] *= postf;
  }
  if (P.act) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int k = 0; k < 4; ++k) acc[j][k] = acc[j][k] > 0.f ? acc[j][k] : acc[j][k] * P.act_slope;
  }
  if (P.self_out) {
#pragma unroll
    for (int j = 0; j < 4; ++j) t[j] = ld_gather4(sc + ((size_t)row * B + bq[j]) * P.ld_src);
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int b = b_base + 4 * j + q;
    if (b < B) {
      const size_t orow = P.out_nm ? (size_t)row * B + b : (size_t)b * n + row;
      if (P.self_out) st4(P.self_out + orow * P.ld_self + sl * 4, t[j]);
      st4(P.out + orow * P.ld_out + sl * 4, make_float4(acc[j][0], acc[j][1], acc[j][2], acc[j][3]));
    }
  }
}

__global__ void edge_values_kernel(const float* __restrict__ ea, const int* __restrict__ eid,
                                   const int* __restrict__ rowptr, int n_rows, long long cap, float fill,
                                   float* __restrict__ val) {
  const long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (q >= cap) return;
  const int nnz = __ldg(rowptr + n_rows);
  float v = 0.f;
  if (q < nnz) {
    const int e = __ldg(eid + q);
    v = e >= 0 ? __ldg(ea + e) : fill;
  }
  val[q] = v;
}

__global__ void embed_scale_fwd_kernel(const float* __restrict__ xs, const float* __restrict__ emb,
                                       long long total4, int N, int C4, float4* __restrict__ out) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const long long r = i / C4;
  const int c4 = (int)(i - r * C4);
  const int n = (int)(r % N);
  const float s = __ldg(xs + r);
  const float4 e = __ldg(reinterpret_cast<const float4*>(emb) + (size_t)n * C4 + c4);
  out[i] = make_float4(s * e.x, s * e.y, s * e.z, s * e.w);
}

__global__ void embed_scale_bwd_kernel(const float* __restrict__ xs, const float4* __restrict__ g, int B,
                                       int N, int C4, float4* __restrict__ g_emb) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= (long long)N * C4) return;
  const int n = (int)(i / C4);
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int b = 0; b < B; ++b) {
    const float s = __ldg(xs + (size_t)b * N + n);
    const float4 v = __ldg(g + (size_t)b * N * C4 + i);
    a.x = fmaf(s, v.x, a.x);
    a.y = fmaf(s, v.y, a.y);
    a.z = fmaf(s, v.z, a.z);
    a.w = fmaf(s, v.w, a.w);
  }
  g_emb[i] = a;
}

// replica slices of the replicated path (grid = row blocks x slices; also the number of partial rows per node that
// the reduce_scale mode writes)
inline int rep_slices(long long gx, long long replicas) {
  int gy = 1;
  static const int cta_target = getenv("MLG_GS_CTAS") ? atoi(getenv("MLG_GS_CTAS")) : 148 * 16;
  while (gx * gy < cta_target && (replicas / (gy * 2)) >= RB) gy *= 2;
  return gy;
}

inline void rep_geometry(int64_t C, bool vec4, int* lanes, int* rows_per_block) {
  const int wpb = kThreads / 32;
  *lanes = 32;
  *rows_per_block = wpb;
  if (vec4 && C <= 32) { *lanes = 8; *rows_per_block = wpb * 4; }
  else if (vec4 && C <= 64) { *lanes = 16; *rows_per_block = wpb * 2; }
}

}  // namespace

extern "C" int64_t mlg_gather_sum_slices(int64_t n_rows, int64_t C, int64_t replicas) {
  if (replicas <= 1 || n_rows <= 0) return 1;
  int lanes, rpb;
  rep_geometry(C, C % 4 == 0, &lanes, &rpb);
  return rep_slices(mlg_ceil_div(n_rows, rpb), replicas);
}

extern "C" int mlg_gather_sum(const float* src, int64_t ld_src, const int32_t* rowptr, const int32_t* idx,
                              const float* val, const float* pre, const float* post, const int32_t* order,
                              int64_t n_rows, int64_t C, int64_t replicas, int64_t rep_rows_src,
                              int64_t rep_rows_pre, int post_mode, int relative, const float* addend,
                              int64_t ld_add, float* out, int64_t ld_out, float* self_out, int64_t ld_self,
                              const float* mask, int64_t ld_mask, float mask_slope, const float* reduce_scale,
                              void* stream) {
  return mlg_gather_sum_act(src, ld_src, rowptr, idx, val, pre, post, order, n_rows, C, replicas, rep_rows_src, rep_rows_pre,
                            post_mode, relative, addend, ld_add, out, ld_out, self_out, ld_self, mask, ld_mask, mask_slope,
                            reduce_scale, 0, 0.f, stream);
}

extern "C" int mlg_gather_sum_act(const float* src, int64_t ld_src, const int32_t* rowptr, const int32_t* idx,
                                  const float* val, const float* pre, const float* post, const int32_t* order,
                                  int64_t n_rows, int64_t C, int64_t replicas, int64_t rep_rows_src,
                                  int64_t rep_rows_pre, int post_mode, int relative, const float* addend,
                                  int64_t ld_add, float* out, int64_t ld_out, float* self_out, int64_t ld_self,
                                  const float* mask, int64_t ld_mask, float mask_slope, const float* reduce_scale,
                                  int act, float act_slope, void* stream) {
  MLG_CHECK_ARG(src && rowptr && idx && out, "mlg_gather_sum: null src/rowptr/idx/out");
  MLG_CHECK_ARG(n_rows >= 0 && n_rows < (1ll << 31) && C > 0 && C < (1ll << 20),
                "mlg_gather_sum: bad sizes n_rows=%lld C=%lld", (long long)n_rows, (long long)C);
  MLG_CHECK_ARG(post_mode >= 0 && post_mode <= 2 && (post_mode != 2 || post), "mlg_gather_sum: bad post_mode");
  MLG_CHECK_ARG(replicas >= 1 && replicas * n_rows < (1ll << 31) && replicas * rep_rows_src < (1ll << 31) &&
                    rep_rows_src >= 0 && rep_rows_pre >= 0,
                "mlg_gather_sum: bad replicas");
  MLG_CHECK_ARG(replicas > 1 || (rep_rows_pre == 0), "mlg_gather_sum: per-replica pre needs replicas > 1");
  MLG_CHECK_ARG(rep_rows_src > 0 || replicas == 1 || (pre && rep_rows_pre > 0),
                "mlg_gather_sum: rep_rows_src == 0 (rank-1 source) needs a per-replica pre");
  MLG_CHECK_ARG(ld_src >= C && ld_out >= C && (!addend || ld_add >= C) && (!self_out || ld_self >= C) &&
                    (!mask || ld_mask >= C),
                "mlg_gather_sum: leading dimension smaller than C");
  if (n_rows == 0) return MLG_OK;
  const bool vec4 = C % 4 == 0 && ld_src % 4 == 0 && ld_out % 4 == 0 && (!addend || ld_add % 4 == 0) &&
                    (!self_out || ld_self % 4 == 0) && ((uintptr_t)src % 16 == 0) && ((uintptr_t)out % 16 == 0) &&
                    (!addend || (uintptr_t)addend % 16 == 0) && (!self_out || (uintptr_t)self_out % 16 == 0) &&
                    (!mask || (ld_mask % 4 == 0 && (uintptr_t)mask % 16 == 0));
  GsP P;
  P.src = src; P.rowptr = rowptr; P.idx = idx; P.val = val; P.pre = pre; P.post = post; P.addend = addend;
  P.order = order; P.out = out; P.self_out = self_out; P.mask = mask; P.ld_mask = (unsigned)ld_mask; P.mask_slope = mask_slope; P.red_scale = reduce_scale;
  P.ld_src = (unsigned)ld_src; P.ld_out = (unsigned)ld_out; P.ld_add = (unsigned)ld_add; P.ld_self = (unsigned)ld_self;
  P.n = (int)n_rows; P.C = (int)C; P.post_mode = post_mode; P.relative = relative;
  P.replicas = (int)replicas; P.rep_rows_src = (unsigned)rep_rows_src; P.rep_rows_pre = (unsigned)rep_rows_pre;
  P.act_slope = act_slope; P.act = act;
  MLG_CHECK_ARG(!act || (replicas > 1 && rep_rows_src > 0 && !relative && !reduce_scale),
                "mlg_gather_sum_act: the fused activation needs the replicated path (replicas > 1, per-replica src), no "
                "relative / reduce_scale");
  cudaStream_t st = (cudaStream_t)stream;
  const int wpb = kThreads / 32;
  int lanes = 32, rows_per_block = wpb;
  if (vec4 && C <= 32) { lanes = 8; rows_per_block = wpb * 4; }
  else if (vec4 && C <= 64) { lanes = 16; rows_per_block = wpb * 2; }
  const long long gx = mlg_ceil_div(n_rows, rows_per_block);
  MLG_CHECK_ARG(!reduce_scale || (replicas > 1 && rep_rows_src > 0 && !relative && !self_out && vec4),
                "mlg_gather_sum: reduce_scale needs the replicated path (replicas > 1, per-replica src), no relative / "
                "self_out, and 16-byte aligned operands with C %% 4 == 0");
  if (replicas > 1) {
    // enough blocks for >= 2 waves of 148 SMs x 8 resident blocks; each slice keeps >= RB replicas
    const int gy = rep_slices(gx, replicas);
    const bool rank1 = rep_rows_src == 0;
    MLG_CHECK_ARG(rank1 || rep_rows_pre == 0, "mlg_gather_sum: per-replica pre is only supported with rep_rows_src == 0");
    const unsigned grid = (unsigned)(gx * gy);
    // (the kernel uses no shared memory and wants the whole L1: with the carve-out forced to 100 % shared memory the gbm-shape
    // aggregation ran 72 -> 86 us, with 0 % the same as the default)
#define MLG_REP(L, V)                                                                        \
  if (rank1) gather_sum_rep_kernel<L, V, true><<<grid, kThreads, 0, st>>>(P, gy);            \
  else if (reduce_scale) gather_sum_rep_kernel<L, V, false, true><<<grid, kThreads, 0, st>>>(P, gy); \
  else gather_sum_rep_kernel<L, V, false><<<grid, kThreads, 0, st>>>(P, gy);
    if (!vec4) { MLG_REP(32, 1) }
    else if (lanes == 8) { MLG_REP(8, 4) }
    else if (lanes == 16) { MLG_REP(16, 4) }
    else { MLG_REP(32, 4) }
#undef MLG_REP
  } else {
    if (!vec4) gather_sum_kernel<32, 1><<<(unsigned)gx, kThreads, 0, st>>>(P);
    else if (lanes == 8) gather_sum_kernel<8, 4><<<(unsigned)gx, kThreads, 0, st>>>(P);
    else if (lanes == 16) gather_sum_kernel<16, 4><<<(unsigned)gx, kThreads, 0, st>>>(P);
    else gather_sum_kernel<32, 4><<<(unsigned)gx, kThreads, 0, st>>>(P);
  }
  MLG_CHECK_LAUNCH("mlg_gather_sum");
  return MLG_OK;
}

extern "C" int mlg_sage_rank1_bwd_rows_supported(int64_t C) { return C == 32 || C == 64; }

static int rank1_bwd_rows_impl(const float* gz, int64_t ld_g, const float* y, const uint64_t* mask_bits, float slope, const float* xs, int xs_transposed, const int32_t* rowptr,
                               const int32_t* idx, const float* val, const int32_t* order, int64_t n_rows,
                               int64_t C, int64_t replicas, float* h, float* g_self, int64_t ld_self,
                               float* g_bias_rows, int gz_node_major, void* stream) {
  MLG_CHECK_ARG(gz && xs && rowptr && idx && h && g_self && g_bias_rows, "mlg_sage_rank1_bwd_rows: null pointer");
  MLG_CHECK_ARG(mlg_sage_rank1_bwd_rows_supported(C), "mlg_sage_rank1_bwd_rows: C=%lld (needs 32 or 64)", (long long)C);
  MLG_CHECK_ARG(n_rows >= 0 && replicas >= 1 && replicas * n_rows < (1ll << 31) && ld_g >= C && ld_self >= C,
                "mlg_sage_rank1_bwd_rows: bad sizes");
  if (n_rows == 0) return MLG_OK;
  R1B P;
  MLG_CHECK_ARG(!mask_bits || C == 64, "mlg_sage_rank1_bwd_rows: mask_bits needs C == 64");
  P.mbits = reinterpret_cast<const unsigned long long*>(mask_bits);
  P.gz = gz; P.y = y; P.slope = slope; P.xs = xs; P.rowptr = rowptr; P.idx = idx; P.val = val; P.order = order; P.h = h; P.g_self = g_self;
  P.g_bias_rows = g_bias_rows; P.ld_g = (unsigned)ld_g; P.ld_self = (unsigned)ld_self; P.n = (int)n_rows; P.B = (int)replicas;
  P.xs_t = xs_transposed; P.gz_nm = gz_node_major;
  const unsigned grid = (unsigned)mlg_ceil_div(n_rows, kThreads / 32);
  cudaStream_t st = (cudaStream_t)stream;
  if (C == 64 && P.xs_t && P.B % 32 == 0) sage_rank1_bwd_rows_kernel<2, true><<<grid, kThreads, 0, st>>>(P);
  else if (C == 64) sage_rank1_bwd_rows_kernel<2, false><<<grid, kThreads, 0, st>>>(P);
  else sage_rank1_bwd_rows_kernel<1, false><<<grid, kThreads, 0, st>>>(P);
  MLG_CHECK_LAUNCH("mlg_sage_rank1_bwd_rows");
  return MLG_OK;
}

extern "C" int mlg_sage_rank1_bwd_rows(const float* gz, int64_t ld_g, const float* y, const uint64_t* mask_bits, float slope, const float* xs, int xs_transposed, const int32_t* rowptr,
                                       const int32_t* idx, const float* val, const int32_t* order, int64_t n_rows,
                                       int64_t C, int64_t replicas, float* h, float* g_self, int64_t ld_self,
                                       float* g_bias_rows, void* stream) {
  return rank1_bwd_rows_impl(gz, ld_g, y, mask_bits, slope, xs, xs_transposed, rowptr, idx, val, order, n_rows, C, replicas, h, g_self,
                             ld_self, g_bias_rows, 0, stream);
}
// gz (and y) with NODE-MAJOR rows, the layout mlg_sage_rank1_fwd_rows_nm writes
extern "C" int mlg_sage_rank1_bwd_rows_nm(const float* gz, int64_t ld_g, const float* y, const uint64_t* mask_bits, float slope, const float* xs, int xs_transposed, const int32_t* rowptr,
                                          const int32_t* idx, const float* val, const int32_t* order, int64_t n_rows,
                                          int64_t C, int64_t replicas, float* h, float* g_self, int64_t ld_self,
                                          float* g_bias_rows, void* stream) {
  return rank1_bwd_rows_impl(gz, ld_g, y, mask_bits, slope, xs, xs_transposed, rowptr, idx, val, order, n_rows, C, replicas, h, g_self,
                             ld_self, g_bias_rows, 1, stream);
}

extern "C" int mlg_edge_values(const float* edge_attr, const int32_t* eid, const int32_t* rowptr,
                               int64_t n_rows, int64_t cap, float fill, float* val, void* stream) {
  MLG_CHECK_ARG(eid && rowptr && val, "mlg_edge_values: null eid/rowptr/val");
  // edge_attr may be NULL when the edge list is empty (every entry is then an added self loop, eid = -1)
  if (cap == 0) return MLG_OK;
  edge_values_kernel<<<mlg_ceil_div(cap, 256), 256, 0, (cudaStream_t)stream>>>(edge_attr, eid, rowptr,
                                                                             (int)n_rows, cap, fill, val);
  MLG_CHECK_LAUNCH("mlg_edge_values");
  return MLG_OK;
}

extern "C" int mlg_embed_scale_fwd(const float* xs, const float* emb, int64_t B, int64_t N, int64_t C,
                                   float* out, void* stream) {
  MLG_CHECK_ARG(xs && emb && out, "mlg_embed_scale_fwd: null pointer");
  MLG_CHECK_ARG(C % 4 == 0 && C > 0, "mlg_embed_scale_fwd: C=%lld must be a multiple of 4", (long long)C);
  const long long total4 = B * N * (C / 4);
  if (total4 == 0) return MLG_OK;
  embed_scale_fwd_kernel<<<mlg_ceil_div(total4, 256), 256, 0, (cudaStream_t)stream>>>(
      xs, emb, total4, (int)N, (int)(C / 4), reinterpret_cast<float4*>(out));
  MLG_CHECK_LAUNCH("mlg_embed_scale_fwd");
  return MLG_OK;
}

extern "C" int mlg_embed_scale_bwd(const float* xs, const float* g_out, int64_t B, int64_t N, int64_t C,
                                   float* g_emb, void* stream) {
  MLG_CHECK_ARG(xs && g_out && g_emb, "mlg_embed_scale_bwd: null pointer");
  MLG_CHECK_ARG(C % 4 == 0 && C > 0, "mlg_embed_scale_bwd: C=%lld must be a multiple of 4", (long long)C);
  const long long total = N * (C / 4);
  if (total == 0) return MLG_OK;
  embed_scale_bwd_kernel<<<mlg_ceil_div(total, 256), 256, 0, (cudaStream_t)stream>>>(
      xs, reinterpret_cast<const float4*>(g_out), (int)B, (int)N, (int)(C / 4),
      reinterpret_cast<float4*>(g_emb));
  MLG_CHECK_LAUNCH("mlg_embed_scale_bwd");
  return MLG_OK;
}

// Replicated aggregation over node-major 32-wide rows (gather_nm_kernel):
//   out_i(b) = act( addend_i(b) + post_i * sum_q val_q * pre[idx_q] * src[idx_q, b] ),  self_out_i(b) = src[i, b]
// src / addend rows node-major (row of (replica b, node j) = j * replicas + b, leading dimensions ld_src / ld_add);
// out / self_out graph-major (b * n_rows + i) or, with out_node_major, node-major too.  post_i = 1 / row length when
// `mean`.  Forward of the transform-first SAGE layer on a node-major [U | V] (SAGEConv.message + mean + update,
// torch_vertex.py:279-291) and its backward aggregation on the by-source CSR.
extern "C" int mlg_gather_sum_nm_ex(const float* src, int64_t ld_src, const int32_t* rowptr, const int32_t* idx, const float* val,
                                    const float* pre, const int32_t* order, int64_t n_rows, int64_t replicas, int mean,
                                    const float* addend, int64_t ld_add, int act, float act_slope, float* out, int64_t ld_out,
                                    float* self_out, int64_t ld_self, int out_node_major, void* stream) {
  MLG_CHECK_ARG(src && rowptr && idx && out, "mlg_gather_sum_nm: null pointer");
  MLG_CHECK_ARG(n_rows >= 0 && replicas >= 1 && replicas * n_rows < (1ll << 31), "mlg_gather_sum_nm: bad sizes");
  MLG_CHECK_ARG(ld_src >= 32 && ld_src % 4 == 0 && ld_out >= 32 && ld_out % 4 == 0 && (!self_out || (ld_self >= 32 && ld_self % 4 == 0)) &&
                    (!addend || (ld_add >= 32 && ld_add % 4 == 0)) &&
                    ((uintptr_t)src | (uintptr_t)out | (uintptr_t)self_out | (uintptr_t)addend) % 16 == 0,
                "mlg_gather_sum_nm: 32-wide rows, 16-byte aligned, leading dimensions multiples of 4");
  if (n_rows == 0) return MLG_OK;
  NmP P;
  P.src = src; P.rowptr = rowptr; P.idx = idx; P.val = val; P.pre = pre; P.order = order; P.addend = addend; P.out = out;
  P.self_out = self_out; P.ld_src = (unsigned)ld_src; P.ld_add = (unsigned)ld_add; P.ld_out = (unsigned)ld_out;
  P.ld_self = (unsigned)ld_self; P.n = (int)n_rows; P.B = (int)replicas; P.mean = mean; P.act = act; P.act_slope = act_slope;
  P.out_nm = out_node_major;
  const long long warps = n_rows * ((replicas + 15) / 16);
  gather_nm_kernel<<<(unsigned)mlg_ceil_div(warps, kThreads / 32), kThreads, 0, (cudaStream_t)stream>>>(P);
  MLG_CHECK_LAUNCH("mlg_gather_sum_nm");
  return MLG_OK;
}

extern "C" int mlg_gather_sum_nm(const float* src, const int32_t* rowptr, const int32_t* idx, const float* val,
                                 const float* pre, const int32_t* order, int64_t n_rows, int64_t replicas, float* out,
                                 int64_t ld_out, float* self_out, int64_t ld_self, void* stream) {
  return mlg_gather_sum_nm_ex(src, 32, rowptr, idx, val, pre, order, n_rows, replicas, 0, nullptr, 0, 0, 0.f, out, ld_out, self_out,
                              ld_self, 0, stream);
}
