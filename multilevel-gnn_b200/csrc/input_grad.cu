// Gradients with respect to the node values x (batch.x) of MultilevelGNN's first layer, and the device-side accumulation
// of per-slot gradients into per-patient attributions (sm_100a).
//
// mlg_sage_rank1_bwd_xs: the fully factored first SAGE layer (csrc/sage_rank1.cu)
//     z[b,i,:] = xs[b,i] E_self[i,:] + (1/cnt_i) sum_{q in row i} val_q xs[b,j_q] E_nbr[j_q,:] + bias,   y = LeakyReLU(z)
// has the input gradient
//     g_xs[b,j] = <gz[b,j,:], E_self[j,:]> + sum_{(i,q): j_q = j} (val_q / cnt_i) <gz[b,i,:], E_nbr[j,:]>.
// It is organised by TARGET row, like mlg_sage_rank1_bwd_rows: one warp per gene i, lane l keeps channels l (and l + 32) of
// 32 replicas' gz rows in registers (gz is read once).  Per CSR entry the warp loads the source's E_nbr row once (the tables
// are L2-resident), forms the 32 replica dot products as per-lane partials, and a butterfly reduce-scatter (31 shuffle+add
// steps) leaves lane b with replica b's sum: one coalesced store of the entry's [B] values.  A second kernel sums the entries
// of every source j over the by-source CSR in a fixed order and adds the self term: deterministic, no atomics.  The
// reduction tree of a replica's dot product does not depend on its slot, so a graph's gradient is the same bits in any slot
// of any batch.
//
// mlg_embed_scale_bwd_xs: g_xs[b,n] = <g_x0[b,n,:], emb[n,:]> for the materialised prologue x0 = xs * emb.
// mlg_attr_accumulate: acc[p,:] (+)= sum_{s in slots of p} w[s] * g[s,:], slots in order (integrated gradients' trapezoid sum).
#include "common.cuh"
#include "../../include/mlg_b200.h"

namespace {

constexpr int kThreads = 256;

// v[32] spread over the warp -> lane l returns the warp-wide sum of v[l] (31 shuffles; fixed tree per value index)
__device__ __forceinline__ float reduce_scatter32(float (&v)[32], int lane) {
  int off = 16;
#pragma unroll
  for (int n = 32; n > 1; n >>= 1, off >>= 1) {
    const bool up = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < n / 2; ++i) {
      const float send = up ? v[i] : v[i + n / 2];
      const float keep = up ? v[i + n / 2] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0];
}

struct R1X {
  const float* gz;
  const float* y;                    // optional: gz is dL/dy; LeakyReLU'(y), y in the layout of gz
  const unsigned long long* mbits;   // optional (C == 64): the forward kernel's sign bits [n][B]
  float slope;
  const float* e_self;
  const float* e_nbr;
  const int* rowptr;
  const int* idx;
  const float* val;
  const int* order;
  float* hx;   // [cap][B]: per-entry values
  float* sx;   // [n][B]: self terms
  unsigned ld_g, ld_self, ld_nbr;
  int n, B;
  int gz_nm;   // gz (and y) rows node-major: (replica b, node i) at i * B + b
};

template <int CPL>
__global__ void __launch_bounds__(kThreads) sage_rank1_bwd_xs_kernel(const R1X P) {
  const int lane = threadIdx.x & 31;
  const long long slot = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (slot >= P.n) return;
  const unsigned row = P.order ? (unsigned)__ldg(P.order + slot) : (unsigned)slot;
  const int beg = __ldg(P.rowptr + row), end = __ldg(P.rowptr + row + 1);
  const float inv = end > beg ? 1.f / (float)(end - beg) : 0.f;
  float es[CPL];
#pragma unroll
  for (int k = 0; k < CPL; ++k) es[k] = __ldg(P.e_self + (size_t)row * P.ld_self + lane + 32 * k);
  for (int rb0 = 0; rb0 < P.B; rb0 += 32) {
    const int nb = min(32, P.B - rb0);
    float g[CPL][32];
    const size_t rstride = P.gz_nm ? (size_t)P.ld_g : (size_t)P.n * P.ld_g;
    const size_t rbase = (P.gz_nm ? (size_t)row * P.B + rb0 : (size_t)rb0 * P.n + row) * P.ld_g + lane;
#pragma unroll
    for (int b = 0; b < 32; ++b)
#pragma unroll
      for (int k = 0; k < CPL; ++k) g[k][b] = b < nb ? __ldg(P.gz + rbase + (size_t)b * rstride + 32 * k) : 0.f;
    if (P.mbits) {   // bit layout of sage_rank1.cu: channel c at bit 16 * (c % 4) + c / 4
      const unsigned long long wd = lane < nb ? __ldg(P.mbits + (size_t)row * P.B + rb0 + lane) : ~0ull;
      const unsigned lo = (unsigned)wd, hi = (unsigned)(wd >> 32);
      const int pos = (lane & 3) * 16 + (lane >> 2);
#pragma unroll
      for (int b = 0; b < 32; ++b) {
        const unsigned long long w =
            ((unsigned long long)__shfl_sync(0xffffffffu, hi, b) << 32) | __shfl_sync(0xffffffffu, lo, b);
        g[0][b] *= ((w >> pos) & 1ull) ? 1.f : P.slope;
        if (CPL == 2) g[CPL - 1][b] *= ((w >> (pos + 8)) & 1ull) ? 1.f : P.slope;
      }
    } else if (P.y) {
#pragma unroll
      for (int b = 0; b < 32; ++b)
#pragma unroll
        for (int k = 0; k < CPL; ++k) {
          const float yv = b < nb ? __ldg(P.y + rbase + (size_t)b * rstride + 32 * k) : 1.f;
          g[k][b] *= yv > 0.f ? 1.f : P.slope;
        }
    }
    {
      float v[32];
#pragma unroll
      for (int b = 0; b < 32; ++b) {
        float d = g[0][b] * es[0];
#pragma unroll
        for (int k = 1; k < CPL; ++k) d = fmaf(g[k][b], es[k], d);
        v[b] = d;
      }
      const float s = reduce_scatter32(v, lane);
      if (lane < nb) P.sx[(size_t)row * P.B + rb0 + lane] = s;
    }
    for (int base = beg; base < end; base += 32) {
      const int q = min(base + lane, end - 1);
      const unsigned my_idx = (unsigned)__ldg(P.idx + q);
      const float my_w = (P.val ? __ldg(P.val + q) : 1.f) * inv;
      const int cnt = min(32, end - base);
      for (int j = 0; j < cnt; ++j) {
        const unsigned src = __shfl_sync(0xffffffffu, my_idx, j);
        const float w = __shfl_sync(0xffffffffu, my_w, j);
        float e[CPL];
#pragma unroll
        for (int k = 0; k < CPL; ++k) e[k] = __ldg(P.e_nbr + (size_t)src * P.ld_nbr + lane + 32 * k);
        float v[32];
#pragma unroll
        for (int b = 0; b < 32; ++b) {
          float d = g[0][b] * e[0];
#pragma unroll
          for (int k = 1; k < CPL; ++k) d = fmaf(g[k][b], e[k], d);
          v[b] = d;
        }
        const float s = reduce_scatter32(v, lane);
        if (lane < nb) P.hx[(size_t)(base + j) * P.B + rb0 + lane] = s * w;
      }
    }
  }
}

// g_xs[b * n + j] = sx[j, b] + sum_{k in by-source row j} hx[fwd_pos[k], b]   (fixed order)
__global__ void rank1_xs_segsum_kernel(const float* __restrict__ hx, const float* __restrict__ sx, const int* __restrict__ rowptr_t,
                                       const int* __restrict__ fwd_pos, int n, int B, float* __restrict__ g_xs) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= (long long)n * B) return;
  const int j = (int)(i / B), b = (int)(i - (long long)j * B);
  float s = __ldg(sx + i);
  const int beg = __ldg(rowptr_t + j), end = __ldg(rowptr_t + j + 1);
  for (int k = beg; k < end; ++k) s += __ldg(hx + (size_t)__ldg(fwd_pos + k) * B + b);
  g_xs[(size_t)b * n + j] = s;
}

__global__ void embed_scale_bwd_xs_kernel(const float* __restrict__ g, const float* __restrict__ emb, long long rows, int N, int C,
                                          float* __restrict__ g_xs) {
  const long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const float* gr = g + (size_t)r * C;
  const float* er = emb + (size_t)(r % N) * C;
  float s = 0.f;
  for (int c = 0; c < C; ++c) s = fmaf(__ldg(gr + c), __ldg(er + c), s);
  g_xs[r] = s;
}

__global__ void attr_accumulate_kernel(const float* __restrict__ g, long long ld_g, const float* __restrict__ w,
                                       const int* __restrict__ slot_ptr, int n_out, long long N, int accumulate,
                                       float* __restrict__ acc) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= (long long)n_out * N) return;
  const int p = (int)(i / N);
  const long long c = i - (long long)p * N;
  float s = accumulate ? acc[i] : 0.f;
  const int beg = __ldg(slot_ptr + p), end = __ldg(slot_ptr + p + 1);
  for (int k = beg; k < end; ++k) s = fmaf(__ldg(w + k), __ldg(g + (size_t)k * ld_g + c), s);
  acc[i] = s;
}

}  // namespace

extern "C" int64_t mlg_sage_rank1_bwd_xs_workspace_bytes(int64_t cap, int64_t n_rows, int64_t replicas) {
  return (cap + n_rows) * replicas * (int64_t)sizeof(float);
}

extern "C" int mlg_sage_rank1_bwd_xs(const float* gz, int64_t ld_g, int gz_node_major, const float* y, const uint64_t* mask_bits,
                                     float slope, const float* e_self, int64_t ld_self, const float* e_nbr, int64_t ld_nbr,
                                     const int32_t* rowptr, const int32_t* idx, const float* val, const int32_t* order,
                                     const int32_t* rowptr_t, const int32_t* fwd_pos_t, int64_t n_rows, int64_t cap, int64_t C,
                                     int64_t replicas, float* g_xs, void* workspace, int64_t workspace_bytes, void* stream) {
  MLG_CHECK_ARG(gz && e_self && e_nbr && rowptr && idx && rowptr_t && fwd_pos_t && g_xs && workspace,
                "mlg_sage_rank1_bwd_xs: null pointer");
  MLG_CHECK_ARG(C == 32 || C == 64, "mlg_sage_rank1_bwd_xs: C=%lld (needs 32 or 64)", (long long)C);
  MLG_CHECK_ARG(!mask_bits || C == 64, "mlg_sage_rank1_bwd_xs: mask_bits needs C == 64");
  MLG_CHECK_ARG(n_rows >= 0 && cap >= 0 && replicas >= 1 && replicas <= 64 && replicas * n_rows < (1ll << 31) &&
                    replicas * cap < (1ll << 31) && ld_g >= C && ld_self >= C && ld_nbr >= C,
                "mlg_sage_rank1_bwd_xs: bad sizes (replicas must be 1..64)");
  MLG_CHECK_ARG(workspace_bytes >= mlg_sage_rank1_bwd_xs_workspace_bytes(cap, n_rows, replicas),
                "mlg_sage_rank1_bwd_xs: workspace too small");
  if (n_rows == 0) return MLG_OK;
  R1X P;
  P.gz = gz; P.y = mask_bits ? nullptr : y; P.mbits = reinterpret_cast<const unsigned long long*>(mask_bits); P.slope = slope;
  P.e_self = e_self; P.e_nbr = e_nbr; P.rowptr = rowptr; P.idx = idx; P.val = val; P.order = order;
  P.hx = static_cast<float*>(workspace);
  P.sx = P.hx + (size_t)cap * replicas;
  P.ld_g = (unsigned)ld_g; P.ld_self = (unsigned)ld_self; P.ld_nbr = (unsigned)ld_nbr;
  P.n = (int)n_rows; P.B = (int)replicas; P.gz_nm = gz_node_major ? 1 : 0;
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned grid = (unsigned)mlg_ceil_div(n_rows, kThreads / 32);
  if (C == 64) sage_rank1_bwd_xs_kernel<2><<<grid, kThreads, 0, st>>>(P);
  else sage_rank1_bwd_xs_kernel<1><<<grid, kThreads, 0, st>>>(P);
  MLG_CHECK_LAUNCH("mlg_sage_rank1_bwd_xs(rows)");
  rank1_xs_segsum_kernel<<<mlg_ceil_div(n_rows * replicas, 256), 256, 0, st>>>(P.hx, P.sx, rowptr_t, fwd_pos_t, (int)n_rows,
                                                                              (int)replicas, g_xs);
  MLG_CHECK_LAUNCH("mlg_sage_rank1_bwd_xs(segsum)");
  return MLG_OK;
}

extern "C" int mlg_embed_scale_bwd_xs(const float* g_out, const float* emb, int64_t B, int64_t N, int64_t C, float* g_xs,
                                      void* stream) {
  MLG_CHECK_ARG(g_out && emb && g_xs, "mlg_embed_scale_bwd_xs: null pointer");
  MLG_CHECK_ARG(B >= 1 && N >= 1 && C >= 1, "mlg_embed_scale_bwd_xs: bad sizes");
  const long long rows = B * N;
  embed_scale_bwd_xs_kernel<<<mlg_ceil_div(rows, 256), 256, 0, (cudaStream_t)stream>>>(g_out, emb, rows, (int)N, (int)C, g_xs);
  MLG_CHECK_LAUNCH("mlg_embed_scale_bwd_xs");
  return MLG_OK;
}

extern "C" int mlg_attr_accumulate(const float* g, int64_t ld_g, const float* w, const int32_t* slot_ptr, int64_t n_out, int64_t N,
                                   int accumulate, float* acc, void* stream) {
  MLG_CHECK_ARG(g && w && slot_ptr && acc, "mlg_attr_accumulate: null pointer");
  MLG_CHECK_ARG(n_out >= 1 && N >= 1 && ld_g >= N && n_out * N < (1ll << 40), "mlg_attr_accumulate: bad sizes");
  attr_accumulate_kernel<<<mlg_ceil_div(n_out * N, 256), 256, 0, (cudaStream_t)stream>>>(g, ld_g, w, slot_ptr, (int)n_out, N,
                                                                                       accumulate, acc);
  MLG_CHECK_LAUNCH("mlg_attr_accumulate");
  return MLG_OK;
}
