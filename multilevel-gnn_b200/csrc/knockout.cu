// Incremental trunk of an in-silico knockout screen for MultilevelGNN (sm_100a).
//
// Setting the values of a node set G to a baseline changes the first SAGE layer only on the rows T1(G) whose CSR entries
// read a node of G (G itself through the self loops), the second layer only on the rows T2(G) that read a T1 row, and
// the pooled features only in the segments that hold a slot of a T2 node (the value mask multiplies by the node's own
// value).  For one work item (patient b, group k) the kernels below recompute exactly those rows, each TWICE --
// with the patient's values and with the knocked-out values -- with the same arithmetic in the same thread, and write
//     pooled'[s, p, c] = pooled_base[b, s, p, c] + sum_{slots q of T2 nodes in segment s} (x2m' - x2m)[node(q), c] w[q, p]
// so a group whose values already equal the baseline leaves pooled' bitwise equal to pooled_base, and a segment no T2
// node reaches is copied unchanged.  No atomics; every sum runs in a fixed order (CSR order, channel order, slot order),
// so an item's output has the same bits whatever its row in the launch and whatever the other items are.
#include "common.cuh"
#include "../../include/mlg_b200.h"

namespace {

constexpr int kC1 = 64;            // first-layer width (hidden_channels of the shipped configs)
constexpr int kC2 = 32;            // second-layer width (final_channels)
constexpr int kWarps = 8;
constexpr int kMaxP = 8;

struct KoP {
  const float *xs, *baseline, *e12, *b1, *wst2, *b2, *uv, *val, *w, *pooled;
  const int32_t *rowptr, *col;
  const int32_t *g_ptr, *g_nodes, *t1_ptr, *t1_nodes, *t2_ptr, *t2_nodes, *s_ptr, *s_seg, *e_ptr, *e_slot, *e_t2;
  const int64_t *item_b, *item_k;
  long long ld_e;
  int N, B, S, P, max_t1, max_t2;
  float slope1, slope2;
  float *uvk, *d2, *out;
};

// position of key in the ascending list a[0..n), or -1
__device__ __forceinline__ int find_sorted(const int32_t* __restrict__ a, int n, int key) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(a + mid) < key) lo = mid + 1;
    else hi = mid;
  }
  return (lo < n && __ldg(a + lo) == key) ? lo : -1;
}

__device__ __forceinline__ float leaky(float z, float slope) { return z > 0.f ? z : z * slope; }

// Layer 1 on the T1 rows of item blockIdx.y, one warp per row, lane = channels 2l, 2l+1:
//   z1 = xs_i E_self[i] + inv_cnt_i sum_j w_ij xs_j E_nbr[j] + b1,  y1 = LeakyReLU(z1),  [U | V] = y1 Wst2^T + [b | 0]
// for the base and the knocked-out values; uvk[r][t][0 / 1][64].
__global__ void __launch_bounds__(kWarps * 32) ko_layer1_kernel(const KoP P) {
  __shared__ __align__(16) float wt[kC1][2 * kC2];      // Wst2^T: lane l reads outputs 2l, 2l+1 of input channel c
  const int r = blockIdx.y;
  const long long k = P.item_k[r];
  if (k < 0) return;
  const int t0 = __ldg(P.t1_ptr + k), nt = __ldg(P.t1_ptr + k + 1) - t0;
  if ((int)blockIdx.x * kWarps >= nt) return;
  for (int q = threadIdx.x; q < kC1 * 2 * kC2; q += blockDim.x) wt[q % kC1][q / kC1] = __ldg(P.wst2 + q);
  __syncthreads();
  const int lane = threadIdx.x & 31, t = blockIdx.x * kWarps + (threadIdx.x >> 5);
  if (t >= nt) return;
  const int b = (int)P.item_b[r];
  const int g0 = __ldg(P.g_ptr + k), ng = __ldg(P.g_ptr + k + 1) - g0;
  const int32_t* gn = P.g_nodes + g0;
  const float* xb = P.xs + (size_t)b * P.N;
  const int i = __ldg(P.t1_nodes + t0 + t);
  const int beg = __ldg(P.rowptr + i), end = __ldg(P.rowptr + i + 1);
  const float inv = end > beg ? 1.f / (float)(end - beg) : 0.f;
  float ab0 = 0.f, ab1 = 0.f, ap0 = 0.f, ap1 = 0.f;
  for (int e0 = beg; e0 < end; e0 += 32) {
    // lane u looks up entry e0 + u (node, weight, both values); the sums then run over the entries in order
    int j = 0;
    float sb = 0.f, sp = 0.f;
    if (e0 + lane < end) {
      j = __ldg(P.col + e0 + lane);
      const float wv = P.val ? __ldg(P.val + e0 + lane) : 1.f;
      const float xj = __ldg(xb + j);
      const float xpj = find_sorted(gn, ng, j) >= 0 ? __ldg(P.baseline + j) : xj;
      sb = wv * xj;
      sp = wv * xpj;
    }
    const int cnt = min(32, end - e0);
#pragma unroll 4
    for (int u = 0; u < cnt; ++u) {
      const int ju = __shfl_sync(0xffffffffu, j, u);
      const float sbu = __shfl_sync(0xffffffffu, sb, u), spu = __shfl_sync(0xffffffffu, sp, u);
      const float2 en = __ldg(reinterpret_cast<const float2*>(P.e12 + (size_t)ju * P.ld_e + kC1 + 2 * lane));
      ab0 = fmaf(sbu, en.x, ab0);
      ab1 = fmaf(sbu, en.y, ab1);
      ap0 = fmaf(spu, en.x, ap0);
      ap1 = fmaf(spu, en.y, ap1);
    }
  }
  const float xi = __ldg(xb + i);
  const float xpi = find_sorted(gn, ng, i) >= 0 ? __ldg(P.baseline + i) : xi;
  const float2 es = __ldg(reinterpret_cast<const float2*>(P.e12 + (size_t)i * P.ld_e + 2 * lane));
  const float bb0 = P.b1 ? __ldg(P.b1 + 2 * lane) : 0.f, bb1 = P.b1 ? __ldg(P.b1 + 2 * lane + 1) : 0.f;
  const float yb0 = leaky(fmaf(es.x, xi, fmaf(ab0, inv, bb0)), P.slope1);
  const float yb1 = leaky(fmaf(es.y, xi, fmaf(ab1, inv, bb1)), P.slope1);
  const float yp0 = leaky(fmaf(es.x, xpi, fmaf(ap0, inv, bb0)), P.slope1);
  const float yp1 = leaky(fmaf(es.y, xpi, fmaf(ap1, inv, bb1)), P.slope1);
  float ub0 = P.b2 ? __ldg(P.b2 + 2 * lane) : 0.f, ub1 = P.b2 ? __ldg(P.b2 + 2 * lane + 1) : 0.f;
  float up0 = ub0, up1 = ub1;
#pragma unroll 8
  for (int q = 0; q < 32; ++q) {           // input channels 2q, 2q + 1, ascending
    const float xb0 = __shfl_sync(0xffffffffu, yb0, q), xb1 = __shfl_sync(0xffffffffu, yb1, q);
    const float xp0 = __shfl_sync(0xffffffffu, yp0, q), xp1 = __shfl_sync(0xffffffffu, yp1, q);
    const float2 w0 = *reinterpret_cast<const float2*>(&wt[2 * q][2 * lane]);
    const float2 w1 = *reinterpret_cast<const float2*>(&wt[2 * q + 1][2 * lane]);
    ub0 = fmaf(xb0, w0.x, ub0); ub1 = fmaf(xb0, w0.y, ub1);
    up0 = fmaf(xp0, w0.x, up0); up1 = fmaf(xp0, w0.y, up1);
    ub0 = fmaf(xb1, w1.x, ub0); ub1 = fmaf(xb1, w1.y, ub1);
    up0 = fmaf(xp1, w1.x, up0); up1 = fmaf(xp1, w1.y, up1);
  }
  float* o = P.uvk + ((size_t)r * P.max_t1 + t) * 2 * (2 * kC2);
  *reinterpret_cast<float2*>(o + 2 * lane) = make_float2(ub0, ub1);
  *reinterpret_cast<float2*>(o + 2 * kC2 + 2 * lane) = make_float2(up0, up1);
}

// Layer 2 on the T2 rows, one warp per row, lane = channel: y2 = LeakyReLU(U_i + inv_cnt_i sum_j w_ij V_j) with U / V from
// layer 1's rows when the node is in T1, else the forward's base row; d2[r][t][c] = y2' x'_i - y2 x_i (the value mask).
__global__ void __launch_bounds__(kWarps * 32) ko_layer2_kernel(const KoP P) {
  const int r = blockIdx.y;
  const long long k = P.item_k[r];
  if (k < 0) return;
  const int t0 = __ldg(P.t2_ptr + k), nt = __ldg(P.t2_ptr + k + 1) - t0;
  const int lane = threadIdx.x & 31, t = blockIdx.x * kWarps + (threadIdx.x >> 5);
  if (t >= nt) return;
  const int b = (int)P.item_b[r];
  const int a0 = __ldg(P.t1_ptr + k), na = __ldg(P.t1_ptr + k + 1) - a0;
  const int32_t* t1n = P.t1_nodes + a0;
  const float* wk = P.uvk + (size_t)r * P.max_t1 * 2 * (2 * kC2);
  const int i = __ldg(P.t2_nodes + t0 + t);
  float Ub, Up;
  const int q = find_sorted(t1n, na, i);
  if (q >= 0) {
    Ub = wk[(size_t)q * 4 * kC2 + lane];
    Up = wk[(size_t)q * 4 * kC2 + 2 * kC2 + lane];
  } else {
    Ub = Up = __ldg(P.uv + ((size_t)i * P.B + b) * (2 * kC2) + lane);
  }
  const int beg = __ldg(P.rowptr + i), end = __ldg(P.rowptr + i + 1);
  const float inv = end > beg ? 1.f / (float)(end - beg) : 0.f;
  float ab = 0.f, ap = 0.f;
  for (int e0 = beg; e0 < end; e0 += 32) {
    // lane u looks up entry e0 + u (node, weight, its row in T1 or -1); the sums then run over the entries in order
    int j = 0, qj = -1;
    float wv = 0.f;
    if (e0 + lane < end) {
      j = __ldg(P.col + e0 + lane);
      wv = P.val ? __ldg(P.val + e0 + lane) : 1.f;
      qj = find_sorted(t1n, na, j);
    }
    const int cnt = min(32, end - e0);
#pragma unroll 2
    for (int u = 0; u < cnt; ++u) {
      const int ju = __shfl_sync(0xffffffffu, j, u), qu = __shfl_sync(0xffffffffu, qj, u);
      const float wu = __shfl_sync(0xffffffffu, wv, u);
      float vb, vp;
      if (qu >= 0) {
        vb = wk[(size_t)qu * 4 * kC2 + kC2 + lane];
        vp = wk[(size_t)qu * 4 * kC2 + 3 * kC2 + lane];
      } else {
        vb = vp = __ldg(P.uv + ((size_t)ju * P.B + b) * (2 * kC2) + kC2 + lane);
      }
      ab = fmaf(wu, vb, ab);
      ap = fmaf(wu, vp, ap);
    }
  }
  const float yb = leaky(fmaf(ab, inv, Ub), P.slope2), yp = leaky(fmaf(ap, inv, Up), P.slope2);
  const int g0 = __ldg(P.g_ptr + k), ng = __ldg(P.g_ptr + k + 1) - g0;
  const float xi = __ldg(P.xs + (size_t)b * P.N + i);
  const float xpi = find_sorted(P.g_nodes + g0, ng, i) >= 0 ? __ldg(P.baseline + i) : xi;
  // explicit roundings: no contraction into an fma, so equal operands give exactly 0
  P.d2[((size_t)r * P.max_t2 + t) * kC2 + lane] = __fsub_rn(__fmul_rn(yp, xpi), __fmul_rn(yb, xi));
}

// Every row of the launch starts as a copy of its patient's base row: out[r] = pooled[item_b[r]] (float4 lanes).
__global__ void __launch_bounds__(256) ko_copy_kernel(const KoP P) {
  const int r = blockIdx.y;
  const size_t n4 = (size_t)P.S * P.P * kC2 / 4;
  const size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= n4) return;
  const float4* src = reinterpret_cast<const float4*>(P.pooled) + (size_t)P.item_b[r] * n4;
  reinterpret_cast<float4*>(P.out)[(size_t)r * n4 + q] = __ldg(src + q);
}

// Then the touched segments of the knockout rows: block (q-th touched segment of item r's group, item r), thread (p, c):
// out = base + sum over the segment's entries, in slot order, of d2[entry's T2 row][c] * w[slot, p].
__global__ void __launch_bounds__(kMaxP * 32) ko_pool_kernel(const KoP P) {
  const int r = blockIdx.y;
  const long long k = P.item_k[r];
  if (k < 0) return;
  const int s0 = __ldg(P.s_ptr + k), ns = __ldg(P.s_ptr + k + 1) - s0;
  const int qs = blockIdx.x;
  if (qs >= ns) return;
  const int p = threadIdx.x >> 5, c = threadIdx.x & 31;
  const int s = __ldg(P.s_seg + s0 + qs);
  const int e0 = __ldg(P.e_ptr + s0 + qs), e1 = __ldg(P.e_ptr + s0 + qs + 1);
  const float* d = P.d2 + (size_t)r * P.max_t2 * kC2 + c;
  float acc = 0.f;
  for (int e = e0; e < e1; ++e)
    acc = fmaf(d[(size_t)__ldg(P.e_t2 + e) * kC2], __ldg(P.w + (size_t)__ldg(P.e_slot + e) * P.P + p), acc);
  if (acc != 0.f) {        // acc == 0 (or -0): the base value itself, bitwise
    const size_t o = ((size_t)s * P.P + p) * kC2 + c;
    P.out[(size_t)r * P.S * P.P * kC2 + o] = __ldg(P.pooled + (size_t)P.item_b[r] * P.S * P.P * kC2 + o) + acc;
  }
}

size_t uvk_floats(int64_t rows, int64_t max_t1) { return (size_t)rows * (size_t)(max_t1 > 0 ? max_t1 : 1) * 4 * kC2; }
size_t d2_floats(int64_t rows, int64_t max_t2) { return (size_t)rows * (size_t)(max_t2 > 0 ? max_t2 : 1) * kC2; }

}  // namespace

extern "C" int64_t mlg_knockout_workspace_bytes(int64_t rows, int64_t max_t1, int64_t max_t2) {
  return (int64_t)(4 * (uvk_floats(rows, max_t1) + d2_floats(rows, max_t2)));
}

extern "C" int mlg_knockout_trunk(const float* xs, const float* baseline, int64_t N, int64_t B, const float* e12, int64_t ld_e12,
                                  const float* b1, float slope1, const float* wst2, const float* b2, const float* uv, float slope2,
                                  const int32_t* rowptr, const int32_t* col, const float* val, const float* w_pool,
                                  const float* pooled, int64_t S, int64_t P, const int32_t* g_ptr, const int32_t* g_nodes,
                                  const int32_t* t1_ptr, const int32_t* t1_nodes, const int32_t* t2_ptr, const int32_t* t2_nodes,
                                  const int32_t* s_ptr, const int32_t* s_seg, const int32_t* e_ptr, const int32_t* e_slot,
                                  const int32_t* e_t2, const int64_t* item_b, const int64_t* item_k, int64_t rows,
                                  int64_t max_t1, int64_t max_t2, void* workspace, int64_t workspace_bytes, float* out,
                                  void* stream) {
  MLG_CHECK_ARG(xs && baseline && e12 && wst2 && uv && rowptr && col && w_pool && pooled && g_ptr && g_nodes && t1_ptr &&
                    t1_nodes && t2_ptr && t2_nodes && s_ptr && s_seg && e_ptr && e_slot && e_t2 && item_b && item_k &&
                    workspace && out,
                "mlg_knockout_trunk: null pointer");
  MLG_CHECK_ARG(N >= 1 && B >= 1 && S >= 1 && rows >= 1 && rows <= 65535 && max_t1 >= 0 && max_t2 >= 0 && N * B < (1ll << 31),
                "mlg_knockout_trunk: bad sizes");
  MLG_CHECK_ARG(P >= 1 && P <= kMaxP, "mlg_knockout_trunk: pca_dim P=%lld outside [1,%d]", (long long)P, kMaxP);
  MLG_CHECK_ARG(((uintptr_t)pooled | (uintptr_t)out) % 16 == 0, "mlg_knockout_trunk: pooled / out must be 16-byte aligned");
  MLG_CHECK_ARG(ld_e12 >= 2 * kC1 && ld_e12 % 2 == 0 && ((uintptr_t)e12 | (uintptr_t)uv) % 8 == 0,
                "mlg_knockout_trunk: e12 must be 8-byte aligned with an even leading dimension >= %d", 2 * kC1);
  MLG_CHECK_ARG(workspace_bytes >= mlg_knockout_workspace_bytes(rows, max_t1, max_t2) && (uintptr_t)workspace % 16 == 0,
                "mlg_knockout_trunk: workspace too small or misaligned");
  KoP p;
  p.xs = xs; p.baseline = baseline; p.e12 = e12; p.b1 = b1; p.wst2 = wst2; p.b2 = b2; p.uv = uv; p.val = val; p.w = w_pool;
  p.pooled = pooled; p.rowptr = rowptr; p.col = col; p.g_ptr = g_ptr; p.g_nodes = g_nodes; p.t1_ptr = t1_ptr;
  p.t1_nodes = t1_nodes; p.t2_ptr = t2_ptr; p.t2_nodes = t2_nodes; p.s_ptr = s_ptr; p.s_seg = s_seg; p.e_ptr = e_ptr;
  p.e_slot = e_slot; p.e_t2 = e_t2; p.item_b = item_b; p.item_k = item_k; p.ld_e = ld_e12;
  p.N = (int)N; p.B = (int)B; p.S = (int)S; p.P = (int)P;
  p.max_t1 = (int)(max_t1 > 0 ? max_t1 : 1); p.max_t2 = (int)(max_t2 > 0 ? max_t2 : 1);
  p.slope1 = slope1; p.slope2 = slope2;
  p.uvk = static_cast<float*>(workspace);
  p.d2 = p.uvk + uvk_floats(rows, max_t1);
  p.out = out;
  cudaStream_t st = (cudaStream_t)stream;
  ko_layer1_kernel<<<dim3((unsigned)mlg_ceil_div(p.max_t1, kWarps), (unsigned)rows), kWarps * 32, 0, st>>>(p);
  MLG_CHECK_LAUNCH("mlg_knockout_trunk (layer 1)");
  ko_layer2_kernel<<<dim3((unsigned)mlg_ceil_div(p.max_t2, kWarps), (unsigned)rows), kWarps * 32, 0, st>>>(p);
  MLG_CHECK_LAUNCH("mlg_knockout_trunk (layer 2)");
  ko_copy_kernel<<<dim3((unsigned)mlg_ceil_div(S * P * kC2 / 4, 256), (unsigned)rows), 256, 0, st>>>(p);
  MLG_CHECK_LAUNCH("mlg_knockout_trunk (copy)");
  ko_pool_kernel<<<dim3((unsigned)S, (unsigned)rows), (unsigned)(P * 32), 0, st>>>(p);
  MLG_CHECK_LAUNCH("mlg_knockout_trunk (pool)");
  return MLG_OK;
}
