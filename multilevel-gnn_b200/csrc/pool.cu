// Gene -> pathway cross-level pool of MultilevelGNN, forward and backward (sm_100a).
//
// Replaces models/multilevel_gnn.py:205-239: value mask (x * batch.x), gather by gene_pca_match,
// missing-gene mask, repeat(P) * (learnable_pca_params * info_mask), permute and
// scatter_reduce(sum) over raw_indice.  The reference materialises [B,C,G,P] fp32 plus an int64 index of
// the same shape (205 MB + 410 MB at the gbm shape) and scatters with atomics; here one warp owns one
// (graph, segment) output row and walks its gene slots, so nothing is materialised and the sum order
// is fixed.  The pooled tensor is produced channel-last, out_cl[b, s, p, c] (lanes run over c: coalesced
// stores, and the 1x1-conv head consumes it as a plain [B*S*P, C] matrix); the reference's
// [B, C, 146, 3P] tensor is a permuted VIEW of it.
// HBM-bound: algorithmic bytes = 4*C*B*N + 4*B*N + 12*G + 4*B*C*S*P  (SURVEY.md section 8d).
#include <cstdlib>

#include "common.cuh"
#include "../../include/mlg_b200.h"

namespace {

constexpr int kThreads = 256;
constexpr int kMaxP = 8;
constexpr int UNP = 8;  // independent row loads in flight per lane

// out_cl[b, s, p, c] = sum_{slot in seg row (b,s)} vm[node] * x[node, c] * w[g, p]
template <int P_>
__global__ void __launch_bounds__(kThreads)
pool_fwd_kernel(const float* __restrict__ x, const float* __restrict__ vm, const long long* __restrict__ match,
                const float* __restrict__ w, const int* __restrict__ rowptr, const int* __restrict__ slots,
                int B, int N, int C, int G, int S, int wrap, float* __restrict__ out_cl) {
  const int lane = threadIdx.x & 31;
  const long long row = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  if (row >= (long long)B * S) return;
  const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
  const long long BN = (long long)B * N;
  for (int c0 = 0; c0 < C; c0 += 32) {
    const int c = c0 + lane;
    const bool cok = c < C;
    float acc[P_];
#pragma unroll
    for (int p = 0; p < P_; ++p) acc[p] = 0.f;
    for (int base = beg; base < end; base += 32) {
      const int q = min(base + lane, end - 1);
      const int slot = __ldg(slots + q);
      const int g = slot % G;
      long long node = __ldg(match + slot);
      float scale = 1.f;
      if (node < 0) {
        if (wrap) node = ((long long)(slot / G) * N + node + BN) % BN;  // python negative index
        else { node = 0; scale = 0.f; }
      } else {
        node += (long long)(slot / G) * N;
      }
      if (vm) scale *= __ldg(vm + node);
      float wl[P_];
#pragma unroll
      for (int p = 0; p < P_; ++p) wl[p] = scale * __ldg(w + (size_t)g * P_ + p);
      const int cnt = min(32, end - base);
      const int inode = (int)node;
      for (int j = 0; j < cnt; j += UNP) {
        float xv[UNP];
#pragma unroll
        for (int u = 0; u < UNP; ++u) {
          const int nj = __shfl_sync(0xffffffffu, inode, min(j + u, cnt - 1));
          xv[u] = cok ? __ldg(x + (size_t)nj * C + c) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < UNP; ++u) {
          const bool on = j + u < cnt;
#pragma unroll
          for (int p = 0; p < P_; ++p) {
            const float wj = __shfl_sync(0xffffffffu, wl[p], min(j + u, cnt - 1));
            acc[p] = fmaf(xv[u], on ? wj : 0.f, acc[p]);
          }
        }
      }
    }
    if (cok) {
      float* o = out_cl + (size_t)row * P_ * C + c;
#pragma unroll
      for (int p = 0; p < P_; ++p) o[(size_t)p * C] = acc[p];
    }
  }
}

// Vector-lane forward for C == 32 * VEC (the shipped widths 32 / 64 / 128): one pass over a segment's slots with
// 64- / 128-bit row loads, UNP rows in flight per lane (v1 above walks the slot list once per 32-channel chunk with
// scalar loads).  VecT / ldvec / stvec are defined with the backward kernels below.
template <int VEC> struct VecF;
template <> struct VecF<1> { typedef float T; };
template <> struct VecF<2> { typedef float2 T; };
template <> struct VecF<4> { typedef float4 T; };

template <int P_, int VEC>
__global__ void __launch_bounds__(kThreads)
pool_fwd_vec_kernel(const float* __restrict__ x, const float* __restrict__ vm, const long long* __restrict__ match,
                    const float* __restrict__ w, const int* __restrict__ rowptr, const int* __restrict__ slots,
                    int B, int N, int G, int S, int wrap, float* __restrict__ out_cl) {
  typedef typename VecF<VEC>::T T;
  constexpr int C = 32 * VEC;
  const int lane = threadIdx.x & 31;
  const long long row = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  if (row >= (long long)B * S) return;
  const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
  const long long BN = (long long)B * N;
  const float* xc = x + lane * VEC;
  float acc[P_][VEC];
#pragma unroll
  for (int p = 0; p < P_; ++p)
#pragma unroll
    for (int k = 0; k < VEC; ++k) acc[p][k] = 0.f;
  for (int base = beg; base < end; base += 32) {
    const int q = min(base + lane, end - 1);
    const int slot = __ldg(slots + q);
    const int g = slot % G;
    long long node = __ldg(match + slot);
    float scale = 1.f;
    if (node < 0) {
      if (wrap) node = ((long long)(slot / G) * N + node + BN) % BN;  // python negative index
      else { node = 0; scale = 0.f; }
    } else {
      node += (long long)(slot / G) * N;
    }
    if (vm) scale *= __ldg(vm + node);
    float wl[P_];
#pragma unroll
    for (int p = 0; p < P_; ++p) wl[p] = scale * __ldg(w + (size_t)g * P_ + p);
    const int cnt = min(32, end - base);
    const int inode = (int)node;
    for (int j = 0; j < cnt; j += UNP) {
      T xv[UNP];
#pragma unroll
      for (int u = 0; u < UNP; ++u) {
        const int nj = __shfl_sync(0xffffffffu, inode, min(j + u, cnt - 1));
        xv[u] = __ldg(reinterpret_cast<const T*>(xc + (size_t)nj * C));
      }
#pragma unroll
      for (int u = 0; u < UNP; ++u) {
        const bool on = j + u < cnt;
        const float* xf = reinterpret_cast<const float*>(&xv[u]);
#pragma unroll
        for (int p = 0; p < P_; ++p) {
          float wj = __shfl_sync(0xffffffffu, wl[p], min(j + u, cnt - 1));
          wj = on ? wj : 0.f;
#pragma unroll
          for (int k = 0; k < VEC; ++k) acc[p][k] = fmaf(xf[k], wj, acc[p][k]);
        }
      }
    }
  }
  float* o = out_cl + (size_t)row * P_ * C + lane * VEC;
#pragma unroll
  for (int p = 0; p < P_; ++p) {
    T t;
    float* tf = reinterpret_cast<float*>(&t);
#pragma unroll
    for (int k = 0; k < VEC; ++k) tf[k] = acc[p][k];
    *reinterpret_cast<T*>(o + (size_t)p * C) = t;
  }
}

// C == 32 forward on 128-bit lanes: an 8-lane group covers one 128-byte row, so a warp has FOUR slots of its segment in
// flight per load instruction (UN4 loads per lane: 32 slots per batch) instead of one; the four groups' partial sums are
// combined with two xor-shuffles per value at the end (fixed order: deterministic).  pool_fwd_vec_kernel<P, 1> walked the
// ~57 slots of a gbm segment in 8 dependent batches of 128-byte loads (36 us for 69 MB); this one needs two.
constexpr int UN4 = 8;
template <int P_>
__global__ void __launch_bounds__(kThreads)
pool_fwd_c32_kernel(const float* __restrict__ x, const float* __restrict__ vm, const long long* __restrict__ match,
                    const float* __restrict__ w, const int* __restrict__ rowptr, const int* __restrict__ slots,
                    int B, int N, int G, int S, int wrap, float* __restrict__ out_cl) {
  constexpr int C = 32;
  const int lane = threadIdx.x & 31;
  const int sub = lane >> 3, sl = lane & 7;
  const long long row = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  if (row >= (long long)B * S) return;
  const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
  const long long BN = (long long)B * N;
  const float* xc = x + sl * 4;
  float acc[P_][4];
#pragma unroll
  for (int p = 0; p < P_; ++p)
#pragma unroll
    for (int k = 0; k < 4; ++k) acc[p][k] = 0.f;
  for (int base = beg; base < end; base += 32) {
    const int q = min(base + lane, end - 1);
    const int slot = __ldg(slots + q);
    const int g = slot % G;
    long long node = __ldg(match + slot);
    float scale = 1.f;
    if (node < 0) {
      if (wrap) node = ((long long)(slot / G) * N + node + BN) % BN;  // python negative index
      else { node = 0; scale = 0.f; }
    } else {
      node += (long long)(slot / G) * N;
    }
    if (vm) scale *= __ldg(vm + node);
    float wl[P_];
#pragma unroll
    for (int p = 0; p < P_; ++p) wl[p] = scale * __ldg(w + (size_t)g * P_ + p);
    const int cnt = min(32, end - base);
    const int inode = (int)node;
    float4 xv[UN4];
#pragma unroll
    for (int u = 0; u < UN4; ++u) {
      if (u * 4 < cnt) {   // warp-uniform
        const int nj = __shfl_sync(0xffffffffu, inode, min(u * 4 + sub, cnt - 1));
        xv[u] = ld_gather4(xc + (size_t)nj * C);
      }
    }
#pragma unroll
    for (int u = 0; u < UN4; ++u) {
      if (u * 4 < cnt) {
        const bool on = u * 4 + sub < cnt;
#pragma unroll
        for (int p = 0; p < P_; ++p) {
          float wj = __shfl_sync(0xffffffffu, wl[p], min(u * 4 + sub, cnt - 1));
          wj = on ? wj : 0.f;
          acc[p][0] = fmaf(xv[u].x, wj, acc[p][0]);
          acc[p][1] = fmaf(xv[u].y, wj, acc[p][1]);
          acc[p][2] = fmaf(xv[u].z, wj, acc[p][2]);
          acc[p][3] = fmaf(xv[u].w, wj, acc[p][3]);
        }
      }
    }
  }
#pragma unroll
  for (int p = 0; p < P_; ++p)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      acc[p][k] += __shfl_xor_sync(0xffffffffu, acc[p][k], 8);
      acc[p][k] += __shfl_xor_sync(0xffffffffu, acc[p][k], 16);
    }
  if (sub == 0) {
    float* o = out_cl + (size_t)row * P_ * C + sl * 4;
#pragma unroll
    for (int p = 0; p < P_; ++p) st4(o + (size_t)p * C, make_float4(acc[p][0], acc[p][1], acc[p][2], acc[p][3]));
  }
}

// g_x[b*N + n, c] = vm * sum_{slot -> node n} sum_p w[g,p] * g_cl[b*S + seg(g), p, c]
// The node-side CSR covers `n_rows` nodes; replicas > 1: one graph's CSR shared by all B graphs
// (gene_pca_match / raw_indice identical for every patient, multiloader.py:697,81-82).
template <int P_>
__global__ void __launch_bounds__(kThreads)
pool_bwd_x_kernel(const float* __restrict__ g_cl, const float* __restrict__ vm, const float* __restrict__ w,
                  const int* __restrict__ rowptr, const int* __restrict__ slots,
                  const int* __restrict__ seg_of_slot, int n_rows, int replicas, int S, int C, int G,
                  float* __restrict__ g_x) {
  constexpr int RB = 8;
  const int lane = threadIdx.x & 31;
  const long long wid = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const int chunks = (replicas + RB - 1) / RB;
  const long long row = wid / chunks;
  const int b0 = (int)(wid % chunks) * RB;
  if (row >= n_rows) return;
  const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
  const size_t rep_g = (size_t)S * P_ * C;  // g_cl elements per replica
  for (int c0 = 0; c0 < C; c0 += 32) {
    const int c = c0 + lane;
    const bool cok = c < C;
    float acc[RB];
#pragma unroll
    for (int r = 0; r < RB; ++r) acc[r] = 0.f;
    for (int base = beg; base < end; base += 32) {
      const int q = min(base + lane, end - 1);
      const int slot = __ldg(slots + q);
      const int g = slot % G;
      const int seg = __ldg(seg_of_slot + slot);  // (b*)S + s
      float wl[P_];
#pragma unroll
      for (int p = 0; p < P_; ++p) wl[p] = __ldg(w + (size_t)g * P_ + p);
      const int cnt = min(32, end - base);
      for (int j = 0; j < cnt; ++j) {
        const int sj = __shfl_sync(0xffffffffu, seg, j);
        float wj[P_];
#pragma unroll
        for (int p = 0; p < P_; ++p) wj[p] = __shfl_sync(0xffffffffu, wl[p], j);
        float gv[RB][P_];
#pragma unroll
        for (int r = 0; r < RB; ++r) {
          const int b = min(b0 + r, replicas - 1);
          const float* gp = g_cl + (size_t)b * rep_g + (size_t)sj * P_ * C + c;
#pragma unroll
          for (int p = 0; p < P_; ++p) gv[r][p] = cok ? __ldg(gp + (size_t)p * C) : 0.f;
        }
#pragma unroll
        for (int r = 0; r < RB; ++r)
#pragma unroll
          for (int p = 0; p < P_; ++p) acc[r] = fmaf(gv[r][p], wj[p], acc[r]);
      }
    }
    if (cok) {
#pragma unroll
      for (int r = 0; r < RB; ++r) {
        const int b = b0 + r;
        if (b < replicas) {
          const size_t orow = (size_t)b * n_rows + row;
          g_x[orow * C + c] = acc[r] * (vm ? __ldg(vm + orow) : 1.f);
        }
      }
    }
  }
}

// g_w[g, p] = sum_b sum_c vm[node] * x[node, c] * g_cl[b*S + seg(b,g), p, c]
// replicated != 0: every graph carries the same match / segment rows (multiloader.py:697), so the slot's node and
// segment are read once and UB graphs' rows are in flight per step.
template <int P_>
__global__ void __launch_bounds__(kThreads)
pool_bwd_w_kernel(const float* __restrict__ g_cl, const float* __restrict__ x, const float* __restrict__ vm,
                  const long long* __restrict__ match, const long long* __restrict__ raw_indice, int B, int N,
                  int C, int G, int S, int wrap, int replicated, float* __restrict__ g_w) {
  constexpr int UB = 8;  // graphs in flight
  const int lane = threadIdx.x & 31;
  const long long g = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  if (g >= G) return;
  const long long BN = (long long)B * N;
  float acc[P_];
#pragma unroll
  for (int p = 0; p < P_; ++p) acc[p] = 0.f;
  const long long m0 = __ldg(match + g), s0 = __ldg(raw_indice + g);
  for (int b0 = 0; b0 < B; b0 += UB) {
    long long node[UB], seg[UB];
    float scale[UB];
#pragma unroll
    for (int u = 0; u < UB; ++u) {
      const int b = min(b0 + u, B - 1);
      long long nd = replicated ? m0 : __ldg(match + (size_t)b * G + g);
      float sc = (b0 + u < B) ? 1.f : 0.f;
      if (nd < 0) {
        if (wrap) nd = ((long long)b * N + nd + BN) % BN;
        else { nd = 0; sc = 0.f; }
      } else {
        nd += (long long)b * N;
      }
      node[u] = nd;
      seg[u] = (long long)b * S + (replicated ? s0 : __ldg(raw_indice + (size_t)b * G + g));
      scale[u] = sc;
    }
    if (vm) {
#pragma unroll
      for (int u = 0; u < UB; ++u) scale[u] *= __ldg(vm + node[u]);
    }
    for (int c = lane; c < C; c += 32) {
      float xv[UB], gv[UB][P_];
#pragma unroll
      for (int u = 0; u < UB; ++u) {
        xv[u] = __ldg(x + (size_t)node[u] * C + c);
#pragma unroll
        for (int p = 0; p < P_; ++p) gv[u][p] = __ldg(g_cl + ((size_t)seg[u] * P_ + p) * C + c);
      }
#pragma unroll
      for (int u = 0; u < UB; ++u) {
        const float xs = xv[u] * scale[u];
#pragma unroll
        for (int p = 0; p < P_; ++p) acc[p] = fmaf(xs, gv[u][p], acc[p]);
      }
    }
  }
#pragma unroll
  for (int p = 0; p < P_; ++p) acc[p] = warp_sum(acc[p]);
  if (lane == 0) {
#pragma unroll
    for (int p = 0; p < P_; ++p) g_w[(size_t)g * P_ + p] = acc[p];
  }
}

// Fused backward: ONE pass over the node-side CSR produces g_x AND per-graph partial weight gradients
//   g_x[b*n + row, c]      = vm * sum_{slot -> row} sum_p w[g,p] * g_cl[b, seg, p, c]
//   part[b, g, p]          = sum_c vm * x[b*n + row, c] * g_cl[b, seg, p, c]          (g = slot's gene)
// x is streamed in node order (coalesced) instead of being gathered per gene slot, and the g_cl rows are loaded
// once for both gradients; g_w = sum_b part[b] is a second, fixed-order pass (deterministic, no atomics).
template <int P_, int CCH, bool WG = true>
__global__ void __launch_bounds__(kThreads)
pool_bwd_fused_kernel(const float* __restrict__ g_cl, const float* __restrict__ x, const float* __restrict__ vm,
                      const float* __restrict__ w, const int* __restrict__ rowptr, const int* __restrict__ slots,
                      const int* __restrict__ seg_of_slot, int n_rows, int replicas, int S, int C, int G,
                      float* __restrict__ g_x, float* __restrict__ part, int mask_input, float mask_slope,
                      float* __restrict__ g_vm) {
  constexpr int RB = 4;
  const int lane = threadIdx.x & 31;
  const long long wid = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const int chunks = (replicas + RB - 1) / RB;
  const long long row = wid / chunks;
  const int b0 = (int)(wid % chunks) * RB;
  if (row >= n_rows) return;
  const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
  const size_t rep_g = (size_t)S * P_ * C;
  float accx[RB][CCH], xr[RB][CCH], scale[RB], dmask[RB][CCH];
#pragma unroll
  for (int r = 0; r < RB; ++r) {
    const int b = min(b0 + r, replicas - 1);
    const size_t orow = (size_t)b * n_rows + row;
    scale[r] = vm ? __ldg(vm + orow) : 1.f;
#pragma unroll
    for (int cc = 0; cc < CCH; ++cc) {
      const int c = cc * 32 + lane;
      accx[r][cc] = 0.f;
      const float raw = (c < C && beg < end) ? __ldg(x + orow * C + c) : 0.f;
      dmask[r][cc] = (mask_input && !(raw > 0.f)) ? mask_slope : 1.f;
      xr[r][cc] = raw * scale[r];
    }
  }
  for (int base = beg; base < end; base += 32) {
    const int q = min(base + lane, end - 1);
    const int slot = __ldg(slots + q);
    const int g = slot % G;
    const int seg = __ldg(seg_of_slot + slot);
    float wl[P_];
#pragma unroll
    for (int p = 0; p < P_; ++p) wl[p] = __ldg(w + (size_t)g * P_ + p);
    const int cnt = min(32, end - base);
    for (int j = 0; j < cnt; ++j) {
      const int sj = __shfl_sync(0xffffffffu, seg, j);
      const int slotj = __shfl_sync(0xffffffffu, slot, j);
      float wj[P_];
#pragma unroll
      for (int p = 0; p < P_; ++p) wj[p] = __shfl_sync(0xffffffffu, wl[p], j);
      float gv[RB][P_][CCH];
#pragma unroll
      for (int r = 0; r < RB; ++r) {
        const int b = min(b0 + r, replicas - 1);
        const float* gp = g_cl + (size_t)b * rep_g + (size_t)sj * P_ * C + lane;
#pragma unroll
        for (int p = 0; p < P_; ++p)
#pragma unroll
          for (int cc = 0; cc < CCH; ++cc) gv[r][p][cc] = (cc * 32 + lane < C) ? __ldg(gp + (size_t)p * C + cc * 32) : 0.f;
      }
#pragma unroll
      for (int r = 0; r < RB; ++r) {
#pragma unroll
        for (int p = 0; p < P_; ++p) {
          float dot = 0.f;
#pragma unroll
          for (int cc = 0; cc < CCH; ++cc) {
            accx[r][cc] = fmaf(gv[r][p][cc], wj[p], accx[r][cc]);
            if constexpr (WG) dot = fmaf(xr[r][cc], gv[r][p][cc], dot);
          }
          if constexpr (WG) {
            dot = warp_sum(dot);
            const int b = b0 + r;
            if (lane == 0 && b < replicas) {
              // replicated layout: slot ids are per graph (part row = b); general layout: slot ids already span b*G + g
              const size_t prow = (replicas > 1) ? (size_t)b * G + slotj : (size_t)slotj;
              part[prow * P_ + p] = dot;
            }
          }
        }
      }
    }
  }
  if (g_vm) {   // dL/dvm = sum_c x * (the unscaled gradient row); x re-read: xr holds it times vm
#pragma unroll
    for (int r = 0; r < RB; ++r) {
      const int b = min(b0 + r, replicas - 1);
      const size_t orow = (size_t)b * n_rows + row;
      float d = 0.f;
#pragma unroll
      for (int cc = 0; cc < CCH; ++cc) {
        const int c = cc * 32 + lane;
        if (c < C && beg < end) d = fmaf(__ldg(x + orow * C + c), accx[r][cc], d);
      }
      d = warp_sum(d);
      if (lane == 0 && b0 + r < replicas) g_vm[orow] = d;
    }
  }
#pragma unroll
  for (int r = 0; r < RB; ++r) {
    const int b = b0 + r;
    if (b >= replicas) continue;
    const size_t orow = (size_t)b * n_rows + row;
#pragma unroll
    for (int cc = 0; cc < CCH; ++cc) {
      const int c = cc * 32 + lane;
      if (c < C) g_x[orow * C + c] = accx[r][cc] * scale[r] * dmask[r][cc];
    }
  }
}

// Second-generation fused backward (C == 32 * VEC, vector lanes, RB2 replicas per warp):
//   * every lane owns VEC consecutive channels (64- / 128-bit loads), the RB2 x-rows of a warp are all requested before
//     anything depends on them, and the g_cl rows of a slot are requested as one batch (min-blocks launch bound so that
//     ptxas keeps them in distinct registers);
//   * the RB2 * P dot products of a slot are reduced across the warp TOGETHER with the packed butterfly (halve the
//     value set at every exchange: K-1+log2(32/K) shuffles for K values instead of 5 per value).
// v1 above spent its time in 40 shuffles + 16 scalar loads per slot (150 us at the gbm shape; HBM floor ~45 us).
template <int K>
__device__ __forceinline__ float reduce_packed(float (&v)[K], int lane) {
  static_assert(K >= 1 && K <= 32 && (K & (K - 1)) == 0, "K must be a power of two <= 32");
  int off = 16;
#pragma unroll
  for (int n = K; n > 1; n >>= 1, off >>= 1) {
    const bool up = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < n / 2; ++i) {
      const float send = up ? v[i] : v[i + n / 2];
      const float keep = up ? v[i + n / 2] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
#pragma unroll
  for (; off >= 1; off >>= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], off);
  return v[0];   // total of value index (lane >> (5 - log2 K)), replicated over the lanes sharing that index
}

template <int VEC> struct VecT;
template <> struct VecT<1> { typedef float T; };
template <> struct VecT<2> { typedef float2 T; };
template <> struct VecT<4> { typedef float4 T; };

template <int VEC>
__device__ __forceinline__ void ldvec(float (&d)[VEC], const float* p) {
  typedef typename VecT<VEC>::T T;
  const T t = __ldg(reinterpret_cast<const T*>(p));
  const float* f = reinterpret_cast<const float*>(&t);
#pragma unroll
  for (int k = 0; k < VEC; ++k) d[k] = f[k];
}
template <int VEC>
__device__ __forceinline__ void stvec(float* p, const float (&d)[VEC]) {
  typedef typename VecT<VEC>::T T;
  T t;
  float* f = reinterpret_cast<float*>(&t);
#pragma unroll
  for (int k = 0; k < VEC; ++k) f[k] = d[k];
  *reinterpret_cast<T*>(p) = t;
}

template <int P_, int VEC, int RB2, bool WG = true>
__global__ void __launch_bounds__(kThreads, (VEC == 1 && RB2 <= 4) ? 4 : 2)
pool_bwd_fused2_kernel(const float* __restrict__ g_cl, const float* __restrict__ x, const float* __restrict__ vm,
                       const float* __restrict__ w, const int* __restrict__ rowptr, const int* __restrict__ slots,
                       const int* __restrict__ seg_of_slot, int n_rows, int replicas, int S, int G,
                       float* __restrict__ g_x, float* __restrict__ part, int mask_input, float mask_slope,
                       float* __restrict__ g_vm) {
  constexpr int C = 32 * VEC;
  constexpr int P2 = P_ <= 1 ? 1 : (P_ <= 2 ? 2 : (P_ <= 4 ? 4 : 8));
  constexpr int K = RB2 * P2;
  constexpr int KSHIFT = K == 1 ? 5 : (K == 2 ? 4 : (K == 4 ? 3 : (K == 8 ? 2 : (K == 16 ? 1 : 0))));
  const int lane = threadIdx.x & 31;
  const long long wid = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const int chunks = (replicas + RB2 - 1) / RB2;
  const long long row = wid / chunks;
  const int b0 = (int)(wid % chunks) * RB2;
  if (row >= n_rows) return;
  const int nb = min(RB2, replicas - b0);
  const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
  const size_t rep_g = (size_t)S * P_ * C;
  const size_t rep_x = (size_t)n_rows * C;
  const unsigned c = lane * VEC;
  float* gx0 = g_x + ((size_t)b0 * n_rows + row) * C + c;
  if (beg == end) {   // node without a gene slot: zero gradient, nothing to read
    float z[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) z[k] = 0.f;
#pragma unroll
    for (int r = 0; r < RB2; ++r)
      if (r < nb) stvec<VEC>(gx0 + (size_t)r * rep_x, z);
    if (g_vm && lane < nb) g_vm[(size_t)(b0 + lane) * n_rows + row] = 0.f;
    return;
  }
  float xr[RB2][VEC], accx[RB2][VEC], scale[RB2];
  const float* x0 = x + ((size_t)b0 * n_rows + row) * C + c;
#pragma unroll
  for (int r = 0; r < RB2; ++r) ldvec<VEC>(xr[r], x0 + (size_t)min(r, nb - 1) * rep_x);
#pragma unroll
  for (int r = 0; r < RB2; ++r) {
    scale[r] = vm ? __ldg(vm + (size_t)(b0 + min(r, nb - 1)) * n_rows + row) : 1.f;
#pragma unroll
    for (int k = 0; k < VEC; ++k) accx[r][k] = 0.f;
  }
  for (int base = beg; base < end; base += 32) {
    const int q = min(base + lane, end - 1);
    const int slot = __ldg(slots + q);
    const int g = slot % G;
    const int seg = __ldg(seg_of_slot + slot);
    float wl[P_];
#pragma unroll
    for (int p = 0; p < P_; ++p) wl[p] = __ldg(w + (size_t)g * P_ + p);
    const int cnt = min(32, end - base);
    for (int j = 0; j < cnt; ++j) {
      const int sj = __shfl_sync(0xffffffffu, seg, j);
      const int slotj = __shfl_sync(0xffffffffu, slot, j);
      float wj[P_];
#pragma unroll
      for (int p = 0; p < P_; ++p) wj[p] = __shfl_sync(0xffffffffu, wl[p], j);
      float gv[RB2][P_][VEC];
      const float* gp = g_cl + (size_t)b0 * rep_g + (size_t)sj * P_ * C + c;
#pragma unroll
      for (int r = 0; r < RB2; ++r)
#pragma unroll
        for (int p = 0; p < P_; ++p) ldvec<VEC>(gv[r][p], gp + (size_t)min(r, nb - 1) * rep_g + (size_t)p * C);
      float d[K];
#pragma unroll
      for (int r = 0; r < RB2; ++r)
#pragma unroll
        for (int p = 0; p < P2; ++p) {
          float dot = 0.f;
          if (p < P_) {
#pragma unroll
            for (int k = 0; k < VEC; ++k) {
              accx[r][k] = fmaf(gv[r][p < P_ ? p : 0][k], wj[p < P_ ? p : 0], accx[r][k]);
              if constexpr (WG) dot = fmaf(xr[r][k], gv[r][p < P_ ? p : 0][k], dot);
            }
          }
          d[r * P2 + p] = dot * scale[r];
        }
      if constexpr (WG) {
        const float tot = reduce_packed<K>(d, lane);
        const int vi = lane >> KSHIFT;
        const int r = vi / P2, p = vi % P2;
        if ((lane & ((1 << KSHIFT) - 1)) == 0 && p < P_ && r < nb) {
          // replicated layout: slot ids are per graph (part row = b); general layout: slot ids already span b*G + g
          const size_t prow = (replicas > 1) ? (size_t)(b0 + r) * G + slotj : (size_t)slotj;
          part[prow * P_ + p] = tot;
        }
      }
    }
  }
  if (g_vm) {   // dL/dvm = sum_c x * (the unscaled gradient row)
#pragma unroll
    for (int r = 0; r < RB2; ++r) {
      float dv = 0.f;
#pragma unroll
      for (int k = 0; k < VEC; ++k) dv = fmaf(xr[r][k], accx[r][k], dv);
      dv = warp_sum(dv);
      if (lane == 0 && r < nb) g_vm[(size_t)(b0 + r) * n_rows + row] = dv;
    }
  }
#pragma unroll
  for (int r = 0; r < RB2; ++r) {
    if (r < nb) {
#pragma unroll
      for (int k = 0; k < VEC; ++k) accx[r][k] *= (mask_input && !(xr[r][k] > 0.f)) ? scale[r] * mask_slope : scale[r];
      stvec<VEC>(gx0 + (size_t)r * rep_x, accx[r]);
    }
  }
}

// C == 32 fused backward on 128-bit lanes: an 8-lane group covers one 128-byte row and owns RBS replicas, so a warp
// covers 4 * RBS replicas of its node with a quarter of the load instructions of pool_bwd_fused2_kernel<P, 1, 4> and half
// as many warps walk the (rowptr -> slot -> segment -> rows) chain; the RBS * P dot products of a slot are reduced inside
// the 8-lane group with the packed butterfly.
template <int K>
__device__ __forceinline__ float reduce_packed8(float (&v)[K], int sl) {
  static_assert(K >= 1 && K <= 8 && (K & (K - 1)) == 0, "K must be a power of two <= 8");
  int off = 4;
#pragma unroll
  for (int n = K; n > 1; n >>= 1, off >>= 1) {
    const bool up = (sl & off) != 0;
#pragma unroll
    for (int i = 0; i < n / 2; ++i) {
      const float send = up ? v[i] : v[i + n / 2];
      const float keep = up ? v[i + n / 2] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
#pragma unroll
  for (; off >= 1; off >>= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], off);
  return v[0];   // total of value index (sl >> (3 - log2 K)), replicated over the lanes sharing that index
}

template <int P_, int RBS, bool WG = true>
__global__ void __launch_bounds__(kThreads, 4)
pool_bwd_c32_kernel(const float* __restrict__ g_cl, const float* __restrict__ x, const float* __restrict__ vm,
                    const float* __restrict__ w, const int* __restrict__ rowptr, const int* __restrict__ slots,
                    const int* __restrict__ seg_of_slot, int n_rows, int replicas, int S, int G,
                    float* __restrict__ g_x, float* __restrict__ part, int mask_input, float mask_slope, int gx_node_major,
                    float* __restrict__ g_vm) {
  constexpr int C = 32;
  constexpr int P2 = P_ <= 1 ? 1 : (P_ <= 2 ? 2 : (P_ <= 4 ? 4 : 8));
  constexpr int KSHIFT = P2 == 1 ? 3 : (P2 == 2 ? 2 : (P2 == 4 ? 1 : 0));
  const int lane = threadIdx.x & 31;
  const int sub = lane >> 3, sl = lane & 7;
  const long long wid = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  constexpr int RW = 4 * RBS;   // replicas per warp
  const int chunks = (replicas + RW - 1) / RW;
  const long long row = wid / chunks;
  if (row >= n_rows) return;
  const int chunk = (int)(wid % chunks);
  const int bs = chunk * RW + sub * RBS;                 // this group's first replica
  const int nb = min(RBS, replicas - bs);                // <= 0: idle group (still takes part in the shuffles)
  const int b0 = nb > 0 ? bs : 0;
  const int nbc = max(nb, 1);
  const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
  const size_t rep_g = (size_t)S * P_ * C;
  const size_t rep_x = (size_t)n_rows * C;
  const unsigned c = sl * 4;
  // gx_node_major: g_x row of (replica b, node i) is i * replicas + b (the replica rows of a node contiguous: what the
  // by-source aggregation that consumes this gradient gathers per CSR entry) instead of b * n_rows + i
  const size_t gx_step = gx_node_major ? (size_t)C : rep_x;
  float* gx0 = g_x + (gx_node_major ? ((size_t)row * replicas + b0) : ((size_t)b0 * n_rows + row)) * C + c;
  if (beg == end) {   // node without a gene slot: zero gradient, nothing to read
#pragma unroll
    for (int r = 0; r < RBS; ++r)
      if (r < nb) st4(gx0 + (size_t)r * gx_step, make_float4(0.f, 0.f, 0.f, 0.f));
    if (g_vm && sl < nb && sl < RBS) g_vm[(size_t)(b0 + sl) * n_rows + row] = 0.f;
    return;
  }
  float4 xr[RBS];
  float accx[RBS][4], scale[RBS];
  const float* x0 = x + ((size_t)b0 * n_rows + row) * C + c;
#pragma unroll
  for (int r = 0; r < RBS; ++r) xr[r] = ld_stream4(x0 + (size_t)min(r, nbc - 1) * rep_x);
#pragma unroll
  for (int r = 0; r < RBS; ++r) {
    scale[r] = vm ? __ldg(vm + (size_t)(b0 + min(r, nbc - 1)) * n_rows + row) : 1.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) accx[r][k] = 0.f;
  }
  for (int base = beg; base < end; base += 32) {
    const int q = min(base + lane, end - 1);
    const int slot = __ldg(slots + q);   // replicated layout: slot ids are per graph (slot < G is the gene slot itself)
    const int seg = __ldg(seg_of_slot + slot);
    float wl[P_];
#pragma unroll
    for (int p = 0; p < P_; ++p) wl[p] = __ldg(w + (size_t)slot * P_ + p);
    const int cnt = min(32, end - base);
    for (int j = 0; j < cnt; ++j) {
      const int sj = __shfl_sync(0xffffffffu, seg, j);
      const int slotj = __shfl_sync(0xffffffffu, slot, j);
      float wj[P_];
#pragma unroll
      for (int p = 0; p < P_; ++p) wj[p] = __shfl_sync(0xffffffffu, wl[p], j);
      float4 gv[RBS][P_];
      const float* gp = g_cl + (size_t)b0 * rep_g + (size_t)sj * P_ * C + c;
#pragma unroll
      for (int r = 0; r < RBS; ++r)
#pragma unroll
        for (int p = 0; p < P_; ++p) gv[r][p] = ld_gather4(gp + (size_t)min(r, nbc - 1) * rep_g + (size_t)p * C);
      // the slot's P weight-gradient terms, summed over this warp's replicas: per group in replica order, the 8 lanes of a
      // group with the packed butterfly, then the four groups (fixed order: deterministic)
      float d[P2];
#pragma unroll
      for (int p = 0; p < P2; ++p) d[p] = 0.f;
#pragma unroll
      for (int r = 0; r < RBS; ++r)
#pragma unroll
        for (int p = 0; p < P_; ++p) {
          const float4 t = gv[r][p];
          accx[r][0] = fmaf(t.x, wj[p], accx[r][0]);
          accx[r][1] = fmaf(t.y, wj[p], accx[r][1]);
          accx[r][2] = fmaf(t.z, wj[p], accx[r][2]);
          accx[r][3] = fmaf(t.w, wj[p], accx[r][3]);
          if constexpr (WG) {
            float dot = xr[r].x * t.x;
            dot = fmaf(xr[r].y, t.y, dot);
            dot = fmaf(xr[r].z, t.z, dot);
            dot = fmaf(xr[r].w, t.w, dot);
            d[p] += r < nb ? dot * scale[r] : 0.f;
          }
        }
      if constexpr (WG) {
        float tot = reduce_packed8<P2>(d, sl);
        tot += __shfl_xor_sync(0xffffffffu, tot, 8);
        tot += __shfl_xor_sync(0xffffffffu, tot, 16);
        const int p = sl >> KSHIFT;
        if (sub == 0 && (sl & ((1 << KSHIFT) - 1)) == 0 && p < P_)
          part[((size_t)chunk * G + slotj) * P_ + p] = tot;   // one partial per (replica chunk, slot): the reduce adds `chunks`
      }
    }
  }
  if (g_vm) {   // dL/dvm = sum_c x * (the unscaled gradient row), summed over the 8 lanes of the group
#pragma unroll
    for (int r = 0; r < RBS; ++r) {
      float dv = xr[r].x * accx[r][0];
      dv = fmaf(xr[r].y, accx[r][1], dv);
      dv = fmaf(xr[r].z, accx[r][2], dv);
      dv = fmaf(xr[r].w, accx[r][3], dv);
      dv += __shfl_xor_sync(0xffffffffu, dv, 1);
      dv += __shfl_xor_sync(0xffffffffu, dv, 2);
      dv += __shfl_xor_sync(0xffffffffu, dv, 4);
      if (sl == 0 && r < nb) g_vm[(size_t)(b0 + r) * n_rows + row] = dv;
    }
  }
#pragma unroll
  for (int r = 0; r < RBS; ++r) {
    if (r < nb) {
      const float xs[4] = {xr[r].x, xr[r].y, xr[r].z, xr[r].w};
#pragma unroll
      for (int k = 0; k < 4; ++k) accx[r][k] *= (mask_input && !(xs[k] > 0.f)) ? scale[r] * mask_slope : scale[r];
      st4(gx0 + (size_t)r * gx_step, make_float4(accx[r][0], accx[r][1], accx[r][2], accx[r][3]));
    }
  }
}

// g_w = sum over the graphs' partials (fixed order); w_mask: the projection weights were w = params * mask[g] (info_mask of
// multilevel_gnn.py:222), so the gradient w.r.t. params is the sum times mask[g] -- no separate elementwise backward pass
__global__ void pool_wgrad_reduce_kernel(const float* __restrict__ part, int B, long long gp, int P, const float* __restrict__ w_mask,
                                         float* __restrict__ g_w) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= gp) return;
  float s = 0.f;
  for (int b = 0; b < B; ++b) s += part[(size_t)b * gp + i];
  g_w[i] = w_mask ? s * __ldg(w_mask + i / P) : s;
}

#define MLG_P_SWITCH(P, CALL)                                           \
  switch (P) {                                                          \
    case 1: { constexpr int P_ = 1; CALL; } break;                      \
    case 2: { constexpr int P_ = 2; CALL; } break;                      \
    case 3: { constexpr int P_ = 3; CALL; } break;                      \
    case 4: { constexpr int P_ = 4; CALL; } break;                      \
    case 5: { constexpr int P_ = 5; CALL; } break;                      \
    case 6: { constexpr int P_ = 6; CALL; } break;                      \
    case 7: { constexpr int P_ = 7; CALL; } break;                      \
    case 8: { constexpr int P_ = 8; CALL; } break;                      \
    default: break;                                                     \
  }

int check_dims(const char* who, int64_t B, int64_t N, int64_t C, int64_t G, int64_t S, int64_t P) {
  MLG_CHECK_ARG(B > 0 && N > 0 && C > 0 && G > 0 && S > 0, "%s: non-positive size", who);
  MLG_CHECK_ARG(P >= 1 && P <= kMaxP, "%s: pca_dim P=%lld outside [1,%d]", who, (long long)P, kMaxP);
  MLG_CHECK_ARG(B * N < (1ll << 31) && B * G < (1ll << 31) && B * S < (1ll << 31), "%s: sizes exceed int32", who);
  return MLG_OK;
}

}  // namespace

extern "C" int mlg_pool_fwd(const float* x, const float* vm, const int64_t* match, const float* w,
                            const int32_t* seg_rowptr, const int32_t* seg_slot, int64_t B, int64_t N,
                            int64_t C, int64_t G, int64_t S, int64_t P, int wrap_negative, float* out_cl,
                            void* stream) {
  MLG_CHECK_ARG(x && match && w && seg_rowptr && seg_slot && out_cl, "mlg_pool_fwd: null pointer");
  int rc = check_dims("mlg_pool_fwd", B, N, C, G, S, P);
  if (rc) return rc;
  const int grid = mlg_ceil_div(B * S, kThreads / 32);
  const bool vec_ok = (C == 32 || C == 64 || C == 128) && (uintptr_t)x % 16 == 0 && (uintptr_t)out_cl % 16 == 0;
#define MLG_POOL_FV(VV)                                                                                        \
  MLG_P_SWITCH(P, (pool_fwd_vec_kernel<P_, VV><<<grid, kThreads, 0, (cudaStream_t)stream>>>(                    \
                      x, vm, (const long long*)match, w, seg_rowptr, seg_slot, (int)B, (int)N, (int)G, (int)S,  \
                      wrap_negative, out_cl)))
  if (vec_ok && C == 32) {
    MLG_P_SWITCH(P, (pool_fwd_c32_kernel<P_><<<grid, kThreads, 0, (cudaStream_t)stream>>>(
                        x, vm, (const long long*)match, w, seg_rowptr, seg_slot, (int)B, (int)N, (int)G, (int)S,
                        wrap_negative, out_cl)));
  }
  else if (vec_ok && C == 64) { MLG_POOL_FV(2); }
  else if (vec_ok) { MLG_POOL_FV(4); }
  else {
    MLG_P_SWITCH(P, (pool_fwd_kernel<P_><<<grid, kThreads, 0, (cudaStream_t)stream>>>(
                        x, vm, (const long long*)match, w, seg_rowptr, seg_slot, (int)B, (int)N, (int)C, (int)G,
                        (int)S, wrap_negative, out_cl)));
  }
#undef MLG_POOL_FV
  MLG_CHECK_LAUNCH("mlg_pool_fwd");
  return MLG_OK;
}

extern "C" int mlg_pool_bwd_x(const float* g_out_cl, const float* vm, const float* w,
                              const int32_t* node_rowptr, const int32_t* node_slot,
                              const int32_t* seg_of_slot, int64_t B, int64_t N, int64_t C, int64_t G,
                              int64_t S, int64_t P, int64_t replicas, float* g_x, void* stream) {
  MLG_CHECK_ARG(g_out_cl && w && node_rowptr && node_slot && seg_of_slot && g_x, "mlg_pool_bwd_x: null pointer");
  int rc = check_dims("mlg_pool_bwd_x", B, N, C, G, S, P);
  if (rc) return rc;
  MLG_CHECK_ARG(replicas == 1 || replicas == B, "mlg_pool_bwd_x: replicas must be 1 or B");
  // replicas == B: the CSR covers one graph (N nodes, G slots, seg ids in [0,S)); else B*N nodes / B*G slots
  const long long n_rows = replicas > 1 ? N : B * N;
  const long long warps = n_rows * ((replicas + 7) / 8);
  const int grid = mlg_ceil_div(warps, kThreads / 32);
  MLG_P_SWITCH(P, (pool_bwd_x_kernel<P_><<<grid, kThreads, 0, (cudaStream_t)stream>>>(
                      g_out_cl, vm, w, node_rowptr, node_slot, seg_of_slot, (int)n_rows, (int)replicas, (int)S,
                      (int)C, (int)G, g_x)));
  MLG_CHECK_LAUNCH("mlg_pool_bwd_x");
  return MLG_OK;
}

extern "C" int mlg_pool_bwd_w(const float* g_out_cl, const float* x, const float* vm, const int64_t* match,
                              const int64_t* raw_indice, int64_t B, int64_t N, int64_t C, int64_t G,
                              int64_t S, int64_t P, int wrap_negative, int64_t replicas, float* g_w, void* stream) {
  MLG_CHECK_ARG(g_out_cl && x && match && raw_indice && g_w, "mlg_pool_bwd_w: null pointer");
  MLG_CHECK_ARG(replicas == 1 || replicas == B, "mlg_pool_bwd_w: replicas must be 1 or B");
  int rc = check_dims("mlg_pool_bwd_w", B, N, C, G, S, P);
  if (rc) return rc;
  const int grid = mlg_ceil_div(G, kThreads / 32);
  MLG_P_SWITCH(P, (pool_bwd_w_kernel<P_><<<grid, kThreads, 0, (cudaStream_t)stream>>>(
                      g_out_cl, x, vm, (const long long*)match, (const long long*)raw_indice, (int)B, (int)N,
                      (int)C, (int)G, (int)S, wrap_negative, replicas > 1 ? 1 : 0, g_w)));
  MLG_CHECK_LAUNCH("mlg_pool_bwd_w");
  return MLG_OK;
}

extern "C" int mlg_pool_bwd_node_major_supported(int64_t C, int64_t replicas) { return C == 32 && replicas > 1; }

extern "C" int mlg_pool_bwd(const float* g_out_cl, const float* x, const float* vm, const float* w,
                            const int32_t* node_rowptr, const int32_t* node_slot, const int32_t* seg_of_slot,
                            int64_t B, int64_t N, int64_t C, int64_t G, int64_t S, int64_t P, int64_t replicas,
                            float* g_x, float* g_w, float* workspace, int mask_input, float mask_slope, const float* w_mask,
                            void* stream) {
  return mlg_pool_bwd_layout(g_out_cl, x, vm, w, node_rowptr, node_slot, seg_of_slot, B, N, C, G, S, P, replicas, g_x, g_w,
                             workspace, mask_input, mask_slope, w_mask, 0, stream);
}

static int pool_bwd_impl(const float* g_out_cl, const float* x, const float* vm, const float* w, const int32_t* node_rowptr,
                         const int32_t* node_slot, const int32_t* seg_of_slot, int64_t B, int64_t N, int64_t C, int64_t G,
                         int64_t S, int64_t P, int64_t replicas, float* g_x, float* g_w, float* workspace, int mask_input,
                         float mask_slope, const float* w_mask, int gx_node_major, float* g_vm, void* stream) {
  MLG_CHECK_ARG(g_out_cl && x && w && node_rowptr && node_slot && seg_of_slot && g_x && (!g_w || workspace),
                "mlg_pool_bwd: null pointer");
  MLG_CHECK_ARG(!gx_node_major || (mlg_pool_bwd_node_major_supported(C, replicas) && (uintptr_t)g_out_cl % 16 == 0 &&
                                   (uintptr_t)x % 16 == 0 && (uintptr_t)g_x % 16 == 0),
                "mlg_pool_bwd_layout: the node-major gradient layout needs C == 32, a replicated layout and 16-byte alignment");
  int rc = check_dims("mlg_pool_bwd", B, N, C, G, S, P);
  if (rc) return rc;
  MLG_CHECK_ARG(replicas == 1 || replicas == B, "mlg_pool_bwd: replicas must be 1 or B");
  MLG_CHECK_ARG(C <= 128, "mlg_pool_bwd: fused backward supports C <= 128 (use mlg_pool_bwd_x / _w)");
  cudaStream_t st = (cudaStream_t)stream;
  const long long n_rows = replicas > 1 ? N : B * N;
  // g_w == NULL: no weight gradient -- the kernels skip the partial dot products, nothing is reduced
  const bool wg = g_w != nullptr;
  static const bool v1_only = getenv("MLG_POOL_BWD_V1") != nullptr;
  if (!v1_only && replicas > 1 && (C == 32 || C == 64 || C == 128) && (uintptr_t)g_out_cl % 16 == 0 && (uintptr_t)x % 16 == 0 &&
      (uintptr_t)g_x % 16 == 0) {
    // vector-lane kernels.  C = 32 has its own kernel (8-lane groups on 128-bit lanes); before it, the 32-lane kernel ran
    // best at 4 replicas per warp (64 registers, 32 warps / SM; 8 per warp: 124 registers / 16 warps, 2 per warp: 48 warps,
    // both slower): the kernel is bound by its dependent loads (rowptr -> slot -> segment -> rows), so resident warps
    // matter more than work per warp.
    if (C == 32) {
      // 8-lane groups x 128-bit lanes: 8 replicas per warp; the weight-gradient partials are already summed over a warp's
      // replicas, so the workspace holds one [G, P] slice per replica chunk (B / 8 of them) instead of one per graph
      constexpr int rw = 8;
      const long long chunks = (replicas + rw - 1) / rw;
      const long long warps3 = n_rows * chunks;
      const int grid3 = mlg_ceil_div(warps3, kThreads / 32);
      if (wg) {
        MLG_CUDA(cudaMemsetAsync(workspace, 0, (size_t)chunks * G * P * sizeof(float), st));   // slots without a node stay zero
        MLG_P_SWITCH(P, (pool_bwd_c32_kernel<P_, 2><<<grid3, kThreads, 0, st>>>(
                            g_out_cl, x, vm, w, node_rowptr, node_slot, seg_of_slot, (int)n_rows, (int)replicas, (int)S,
                            (int)G, g_x, workspace, mask_input, mask_slope, gx_node_major, g_vm)));
      } else {
        MLG_P_SWITCH(P, (pool_bwd_c32_kernel<P_, 2, false><<<grid3, kThreads, 0, st>>>(
                            g_out_cl, x, vm, w, node_rowptr, node_slot, seg_of_slot, (int)n_rows, (int)replicas, (int)S,
                            (int)G, g_x, nullptr, mask_input, mask_slope, gx_node_major, g_vm)));
      }
      MLG_CHECK_LAUNCH("mlg_pool_bwd(c32)");
      if (wg) {
        pool_wgrad_reduce_kernel<<<mlg_ceil_div(G * P, 256), 256, 0, st>>>(workspace, (int)chunks, G * P, (int)P, w_mask, g_w);
        MLG_CHECK_LAUNCH("mlg_pool_bwd(reduce)");
      }
      return MLG_OK;
    }
    if (wg) MLG_CUDA(cudaMemsetAsync(workspace, 0, (size_t)B * G * P * sizeof(float), st));   // slots without a node stay zero
    // C = 64 / 128: replicas per warp chosen so that RB2 * pow2(P) <= 32 packed dot products
    const int rb2 = P <= 4 ? 8 : 4;
    const long long warps2 = n_rows * ((replicas + rb2 - 1) / rb2);
    const int grid2 = mlg_ceil_div(warps2, kThreads / 32);
#define MLG_POOL_F2(VV, RR, WW)                                                                                       \
  MLG_P_SWITCH(P, (pool_bwd_fused2_kernel<P_, VV, RR, WW><<<grid2, kThreads, 0, st>>>(                                 \
                      g_out_cl, x, vm, w, node_rowptr, node_slot, seg_of_slot, (int)n_rows, (int)replicas, (int)S,     \
                      (int)G, g_x, workspace, mask_input, mask_slope, g_vm)))
    if (C == 64 && wg) { MLG_POOL_F2(2, (P_ <= 4 ? 8 : 4), true); }
    else if (C == 64) { MLG_POOL_F2(2, (P_ <= 4 ? 8 : 4), false); }
    else if (wg) { MLG_POOL_F2(4, (P_ <= 4 ? 8 : 4), true); }
    else { MLG_POOL_F2(4, (P_ <= 4 ? 8 : 4), false); }
#undef MLG_POOL_F2
    MLG_CHECK_LAUNCH("mlg_pool_bwd(fused2)");
    if (wg) {
      pool_wgrad_reduce_kernel<<<mlg_ceil_div(G * P, 256), 256, 0, st>>>(workspace, (int)B, G * P, (int)P, w_mask, g_w);
      MLG_CHECK_LAUNCH("mlg_pool_bwd(reduce)");
    }
    return MLG_OK;
  }
  if (wg) MLG_CUDA(cudaMemsetAsync(workspace, 0, (size_t)B * G * P * sizeof(float), st));   // slots without a node stay zero
  const long long warps = n_rows * ((replicas + 3) / 4);
  const int grid = mlg_ceil_div(warps, kThreads / 32);
  const int cch = C <= 32 ? 1 : (C <= 64 ? 2 : 4);
#define MLG_POOL_FUSED(CC, WW)                                                                                         \
  MLG_P_SWITCH(P, (pool_bwd_fused_kernel<P_, CC, WW><<<grid, kThreads, 0, st>>>(g_out_cl, x, vm, w, node_rowptr, node_slot, \
                                                                                seg_of_slot, (int)n_rows, (int)replicas,   \
                                                                                (int)S, (int)C, (int)G, g_x, workspace,   \
                                                                                mask_input, mask_slope, g_vm)))
  if (cch == 1 && wg) { MLG_POOL_FUSED(1, true); }
  else if (cch == 1) { MLG_POOL_FUSED(1, false); }
  else if (cch == 2 && wg) { MLG_POOL_FUSED(2, true); }
  else if (cch == 2) { MLG_POOL_FUSED(2, false); }
  else if (wg) { MLG_POOL_FUSED(4, true); }
  else { MLG_POOL_FUSED(4, false); }
#undef MLG_POOL_FUSED
  MLG_CHECK_LAUNCH("mlg_pool_bwd(fused)");
  if (wg) {
    pool_wgrad_reduce_kernel<<<mlg_ceil_div(G * P, 256), 256, 0, st>>>(workspace, (int)B, G * P, (int)P, w_mask, g_w);
    MLG_CHECK_LAUNCH("mlg_pool_bwd(reduce)");
  }
  return MLG_OK;
}

extern "C" int mlg_pool_bwd_layout(const float* g_out_cl, const float* x, const float* vm, const float* w,
                                   const int32_t* node_rowptr, const int32_t* node_slot, const int32_t* seg_of_slot,
                                   int64_t B, int64_t N, int64_t C, int64_t G, int64_t S, int64_t P, int64_t replicas,
                                   float* g_x, float* g_w, float* workspace, int mask_input, float mask_slope,
                                   const float* w_mask, int gx_node_major, void* stream) {
  MLG_CHECK_ARG(g_w && workspace, "mlg_pool_bwd: null pointer");
  return pool_bwd_impl(g_out_cl, x, vm, w, node_rowptr, node_slot, seg_of_slot, B, N, C, G, S, P, replicas, g_x, g_w, workspace,
                       mask_input, mask_slope, w_mask, gx_node_major, nullptr, stream);
}

extern "C" int mlg_pool_bwd_vm(const float* g_out_cl, const float* x, const float* vm, const float* w,
                               const int32_t* node_rowptr, const int32_t* node_slot, const int32_t* seg_of_slot,
                               int64_t B, int64_t N, int64_t C, int64_t G, int64_t S, int64_t P, int64_t replicas,
                               float* g_x, float* g_w, float* workspace, int mask_input, float mask_slope,
                               const float* w_mask, int gx_node_major, float* g_vm, void* stream) {
  MLG_CHECK_ARG(vm && g_vm, "mlg_pool_bwd_vm: vm and g_vm are required");
  return pool_bwd_impl(g_out_cl, x, vm, w, node_rowptr, node_slot, seg_of_slot, B, N, C, G, S, P, replicas, g_x, g_w, workspace,
                       mask_input, mask_slope, w_mask, gx_node_major, g_vm, stream);
}
