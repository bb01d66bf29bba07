// Metrics of one evaluation split in one kernel (sm_100a): BCE, accuracy and ROC AUC of pred [n, 2] against the one-hot
// target y [n, 2] -- what the reference's eval() computes after its forward-only pass (train.py:71-109).
//
//   bce = torch.nn.BCELoss(weight)(pred, y), mean over all 2n elements, each log clamped at -100, weight = the class row w[c]
//   acc = fraction of rows with argmax(pred) == argmax(y)              (a tie goes to index 0, like torch.argmax)
//   auc = roc_auc_score(argmax(y), pred[:, 1]) as the exact Mann-Whitney count: 2 per positive/negative pair with
//         s_pos > s_neg, 1 per tie, summed in 64-bit integers, over 2 P N (NaN when the split holds one class only)
//
// Every block owns a fixed 256-row tile i of the split and compares its positives with ALL negatives j (the negatives' scores
// stream through shared memory, a positive's slot holds NaN so that it never counts).  Pair, positive and hit counts are
// integer atomics (order-free); the per-element BCE terms are summed per tile in a fixed tree, the tile sums in tile order by
// the last block to finish.  Results are therefore bit-identical from run to run, for any n.  O(n^2) pairs: n <= 65 536.
#include <math.h>

#include "common.cuh"
#include "../../include/mlg_b200.h"

namespace {

constexpr int kTile = 256;          // rows per block (threads per block)
constexpr int kChunk = 2048;        // negatives' scores staged in shared memory per pass
constexpr int64_t kMaxRows = 65536;

struct Header {                     // zeroed before the launch
  unsigned long long pairs;         // Mann-Whitney count (2 per win, 1 per tie)
  unsigned long long pos;           // rows with argmax(y) == 1
  unsigned long long hits;          // rows with argmax(pred) == argmax(y)
  unsigned int ticket;              // blocks done
  unsigned int pad;
};

__device__ __forceinline__ int argmax2(float a, float b) {
  // torch.argmax: NaN is the maximum, the first of equal maxima wins
  if (isnan(a)) return 0;
  if (isnan(b)) return 1;
  return b > a ? 1 : 0;
}

__device__ __forceinline__ double bce_term(float p, float t, float w) {
  // aten binary_cross_entropy: (t - 1) * max(log1p(-p), -100) - t * max(log(p), -100), times the weight
  const float l1 = fmaxf(log1pf(-p), -100.f), l0 = fmaxf(logf(p), -100.f);
  return (double)(w * ((t - 1.f) * l1 - t * l0));
}

__global__ void __launch_bounds__(kTile)
eval_metrics_kernel(const float* __restrict__ pred, const float* __restrict__ y, int n, const float* __restrict__ class_w,
                    Header* __restrict__ hdr, double* __restrict__ tile_bce, float* __restrict__ out) {
  __shared__ float neg[kChunk];
  __shared__ double red_d[kTile / 32];
  __shared__ unsigned long long red_u[3][kTile / 32];
  __shared__ bool last;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int i = blockIdx.x * kTile + tid;
  const float w0 = class_w ? class_w[0] : 1.f, w1 = class_w ? class_w[1] : 1.f;

  float si = 0.f;
  int pos_i = 0, hit = 0;
  double bce = 0.0;
  if (i < n) {
    const float p0 = pred[2 * i], p1 = pred[2 * i + 1], t0 = y[2 * i], t1 = y[2 * i + 1];
    pos_i = argmax2(t0, t1);
    hit = argmax2(p0, p1) == pos_i;
    si = p1;
    bce = bce_term(p0, t0, w0) + bce_term(p1, t1, w1);
  }

  // positives of this tile against every negative of the split
  unsigned int cnt = 0;           // <= 2 * 65 536
  for (int j0 = 0; j0 < n; j0 += kChunk) {
    __syncthreads();
    for (int j = tid; j < kChunk; j += kTile) {
      const int jj = j0 + j;
      float s = __int_as_float(0x7fc00000);          // NaN: never > and never ==
      if (jj < n && argmax2(y[2 * jj], y[2 * jj + 1]) == 0) s = pred[2 * jj + 1];
      neg[j] = s;
    }
    __syncthreads();
    if (i < n && pos_i) {
      const int m = min(kChunk, n - j0);
#pragma unroll 8
      for (int j = 0; j < m; ++j) {
        const float sj = neg[j];
        cnt += (si > sj ? 2u : 0u) + (si == sj ? 1u : 0u);
      }
    }
  }

  // block reductions: integers in any order, the BCE terms in a fixed tree (warp shuffles, then warps in order)
  unsigned long long u0 = cnt, u1 = pos_i, u2 = hit;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    u0 += __shfl_xor_sync(0xffffffffu, u0, o);
    u1 += __shfl_xor_sync(0xffffffffu, u1, o);
    u2 += __shfl_xor_sync(0xffffffffu, u2, o);
    bce += __shfl_xor_sync(0xffffffffu, bce, o);
  }
  if (lane == 0) {
    red_u[0][wid] = u0;
    red_u[1][wid] = u1;
    red_u[2][wid] = u2;
    red_d[wid] = bce;
  }
  __syncthreads();
  if (tid == 0) {
    unsigned long long a = 0, b = 0, c = 0;
    double s = 0.0;
    for (int w = 0; w < kTile / 32; ++w) {
      a += red_u[0][w];
      b += red_u[1][w];
      c += red_u[2][w];
      s += red_d[w];
    }
    atomicAdd(&hdr->pairs, a);
    atomicAdd(&hdr->pos, b);
    atomicAdd(&hdr->hits, c);
    tile_bce[blockIdx.x] = s;
    __threadfence();
    last = atomicAdd(&hdr->ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last || tid != 0) return;
  __threadfence();
  // the last block: tile sums in tile order, then the three metrics
  double s = 0.0;
  for (unsigned b = 0; b < gridDim.x; ++b) s += *(volatile double*)(tile_bce + b);
  const unsigned long long pairs = *(volatile unsigned long long*)&hdr->pairs;
  const unsigned long long P = *(volatile unsigned long long*)&hdr->pos;
  const unsigned long long hits = *(volatile unsigned long long*)&hdr->hits;
  const unsigned long long N = (unsigned long long)n - P;
  out[0] = (float)(s / (2.0 * (double)n));
  out[1] = (float)((double)hits / (double)n);
  out[2] = (P == 0 || N == 0) ? __int_as_float(0x7fc00000) : (float)((double)pairs / (2.0 * (double)P * (double)N));
}

inline int64_t n_tiles(int64_t n) { return (n + kTile - 1) / kTile; }

}  // namespace

extern "C" int64_t mlg_eval_metrics_workspace_bytes(int64_t n) {
  return (int64_t)sizeof(Header) + 8 * (n_tiles(n) < 1 ? 1 : n_tiles(n));
}

extern "C" int mlg_eval_metrics(const float* pred, const float* y, int64_t n, const float* class_w, float* out, void* ws,
                                int64_t ws_bytes, void* stream) {
  MLG_CHECK_ARG(pred && y && out && ws, "mlg_eval_metrics: null pointer");
  MLG_CHECK_ARG(n >= 1 && n <= kMaxRows, "mlg_eval_metrics: need 1 <= n <= %lld (O(n^2) pair count), got %lld",
                (long long)kMaxRows, (long long)n);
  MLG_CHECK_ARG(ws_bytes >= mlg_eval_metrics_workspace_bytes(n), "mlg_eval_metrics: workspace too small");
  MLG_CHECK_ARG((uintptr_t)ws % 8 == 0, "mlg_eval_metrics: workspace must be 8-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  Header* hdr = (Header*)ws;
  MLG_CUDA(cudaMemsetAsync(hdr, 0, sizeof(Header), st));
  eval_metrics_kernel<<<(unsigned)n_tiles(n), kTile, 0, st>>>(pred, y, (int)n, class_w, hdr,
                                                             (double*)((char*)ws + sizeof(Header)), out);
  MLG_CHECK_LAUNCH("mlg_eval_metrics");
  return MLG_OK;
}
