// Pathway Shapley values through MultilevelGNN's head, incrementally along permutations of the players (sm_100a).
//
// The head's input is the pooled grid [32, Hg, Wg] (Hg = 146 pathways, Wg = 3 * pca_dim); its 1x1 convs act on every cell
// alone, so the caller passes per-cell tables c[row][ch * cells + cell] = ReLU(conv2(ReLU(conv1(cell)))) (64 channels, the
// layout mlg_head_conv_pool_fwd writes with a 1x1 window) for the patients and for the background rows.  A (kh, kw)
// floor-mode max-pool window w takes the channel-wise max of its cells, and the first Linear is linear in those maxima:
//     h = b1 + W1[:, age] * age + sum_w W1p[w]^T a0(w),      W1p [Ho * Wo][64][H] (W1 packed by window)
//     p = sigmoid((W3[t] - W3[1-t]) . ReLU(h) + b3[t] - b3[1-t])   (= softmax(W3 ReLU(h) + b3)[t])
// A chain walks one permutation of the players with one patient and one background row j: it starts with every player's
// cells from row j (cells of no player stay the patient's) and adds the players one by one.  Adding player k changes only
// the windows that hold its cells, so a step is h += W1p[w]^T (a0_new(w) - a0_old(w)) over those windows and p costs
// 2 * H FMA.  contrib[chain, k] = p after k - p before k.
//
// One CTA owns kC chains that share one permutation (different patients and / or background rows): one read of a W1p slice
// serves all of them, and the coalition (the players added so far) is the CTA's.  Thread i holds h[i] of every chain in
// registers (blockDim = H).  A window difference of exactly 0 leaves h unchanged, so a player that does not change the grid
// gets exactly 0.  No atomics: every sum has a fixed order that does not depend on the other chains of the CTA.
#include <cmath>

#include "common.cuh"
#include "../../include/mlg_b200.h"

namespace {

constexpr int kC = 16;            // chains per CTA
constexpr int kWT = 4;            // windows per tile of a step (a player may hold one window or a third of them)
constexpr int kCh = 64;           // channels of the second conv
constexpr int kMaxCells = 4096;   // owner table in shared memory (146 x 9 = 1314 for the shipped configs)
constexpr int kMaxWords = 32;     // coalition bitmask: K <= 1024 players

struct ShapP {
  const float *pat, *bg;   // per-cell tables [n_pat][ld], [M][ld]
  long long ld, n_pat, M;
  int Hg, Wg, kh, kw, Wo, nwin, cells;
  const float *w1p, *b1, *w1age, *age, *w3, *b3;
  int target, H;
  const int *owner, *win_ptr, *win_idx;
  int K;
  const int* perm;          // [G][K]
  long long G, n_cp;        // permutations; chains per permutation
  const int *chain_pat, *chain_bg;   // [n_cp], [G][n_cp]
  int tiles;                // CTAs per permutation
  float *contrib, *p0, *pT;
  int* bad;
};

struct Smem {
  float d[kWT * kCh][kC];   // a0 (start) or a0 differences (steps) of the current tile, [row = wt * 64 + ch][chain]
  float red[16][kC];
  float p[kC];
  long long prow[kC], brow[kC];   // element offsets of the chain's patient / background table rows
  float age[kC];
  unsigned coal[kMaxWords];
  int owner[kMaxCells];
};

__device__ __forceinline__ bool in_coal(const Smem& S, int o) { return o < 0 || ((S.coal[o >> 5] >> (o & 31)) & 1u); }

// max over the window's cells of the selected table (patient if the cell's owner is in the coalition, else background),
// starting at 0 as the head does (the values are post-ReLU); with `k` >= 0 also the selection where k has joined.
__device__ __forceinline__ void window_max(const ShapP& P, const Smem& S, int w, int ch, int c, int k, float& old_m,
                                           float& new_m) {
  const float* pr = P.pat + S.prow[c] + (long long)ch * P.cells;
  const float* br = P.bg + S.brow[c] + (long long)ch * P.cells;
  const int ho = w / P.Wo, wo = w - ho * P.Wo;
  float a = 0.f, b = 0.f;
  for (int dh = 0; dh < P.kh; ++dh)
    for (int dw = 0; dw < P.kw; ++dw) {
      const int cell = (ho * P.kh + dh) * P.Wg + wo * P.kw + dw;
      const int o = S.owner[cell];
      const float vp = __ldg(pr + cell);
      const bool sel = in_coal(S, o);
      a = fmaxf(a, sel ? vp : __ldg(br + cell));
      b = fmaxf(b, (sel || o == k) ? vp : __ldg(br + cell));
    }
  old_m = a;
  new_m = b;
}

// h[c] += sum_ch W1p[w][ch][i] * S.d[wt * 64 + ch][c], channels in order; chains in packed pairs (fma.rn.f32x2 is
// IEEE-identical to two fmaf)
__device__ __forceinline__ void window_fma(const ShapP& P, const Smem& S, int wt, int w, u64 (&h)[kC / 2]) {
  const float* rows = P.w1p + (size_t)w * kCh * P.H + threadIdx.x;
#pragma unroll 4
  for (int r = 0; r < kCh; ++r) {
    const float wv = __ldg(rows + (size_t)r * P.H);
    const u64 ww = pk2(wv, wv);
    const ulonglong2* d = reinterpret_cast<const ulonglong2*>(S.d[wt * kCh + r]);
#pragma unroll
    for (int q = 0; q < kC / 4; ++q) {
      const ulonglong2 v = d[q];
      h[2 * q] = fma2(ww, v.x, h[2 * q]);
      h[2 * q + 1] = fma2(ww, v.y, h[2 * q + 1]);
    }
  }
}

// p[c] = sigmoid(dW3 . ReLU(h[c]) + db3): per-warp butterfly sums, then the warps in order (fixed for every chain)
__device__ __forceinline__ void chain_probs(const ShapP& P, Smem& S, float dw3, const u64 (&h)[kC / 2]) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int q = 0; q < kC / 2; ++q) {
    float lo, hi;
    upk2(h[q], lo, hi);
    lo = warp_sum(dw3 * fmaxf(lo, 0.f));
    hi = warp_sum(dw3 * fmaxf(hi, 0.f));
    if (lane == 0) {
      S.red[wid][2 * q] = lo;
      S.red[wid][2 * q + 1] = hi;
    }
  }
  __syncthreads();
  if (threadIdx.x < kC) {
    float z = __ldg(P.b3 + P.target) - __ldg(P.b3 + 1 - P.target);
    for (int q = 0; q < nw; ++q) z += S.red[q][threadIdx.x];
    S.p[threadIdx.x] = 1.f / (1.f + expf(-z));
  }
  __syncthreads();
}

__global__ void __launch_bounds__(512) shap_chains_kernel(const ShapP P) {
  extern __shared__ __align__(16) unsigned char shap_smem[];
  Smem& S = *reinterpret_cast<Smem*>(shap_smem);
  const int i = threadIdx.x;
  const long long g = blockIdx.x / P.tiles;
  const long long s0 = (long long)(blockIdx.x % P.tiles) * kC;
  for (int t = i; t < P.cells; t += blockDim.x) S.owner[t] = __ldg(P.owner + t);
  for (int t = i; t < kMaxWords; t += blockDim.x) S.coal[t] = 0u;
  // chain states: 0 = no chain in this slot, 1 = live, 2 = live with an index outside its table (not read; outputs NaN)
  __shared__ int state[kC];
  if (i < kC) {
    const long long s = s0 + i;
    int st = 0;
    long long pr = -1, br = -1;
    float ag = 0.f;
    if (s < P.n_cp) {
      const int p = __ldg(P.chain_pat + s), j = __ldg(P.chain_bg + g * P.n_cp + s);
      if (p < 0 || p >= P.n_pat || j < 0 || j >= P.M) {
        st = 2;
        *P.bad = 1;
      } else {
        st = 1;
        pr = (long long)p * P.ld;
        br = (long long)j * P.ld;
        ag = P.age ? __ldg(P.age + p) : 0.f;
      }
    }
    state[i] = st;
    S.prow[i] = pr < 0 ? 0 : pr;
    S.brow[i] = br < 0 ? 0 : br;
    S.age[i] = ag;
  }
  __syncthreads();

  // start state: a0 of every window with every player's cells from the background row, one pass over W1p
  u64 h[kC / 2];
  {
    const float b1 = __ldg(P.b1 + i), wa = P.w1age ? __ldg(P.w1age + i) : 0.f;
#pragma unroll
    for (int q = 0; q < kC / 2; ++q)
      h[q] = P.w1age ? pk2(fmaf(wa, S.age[2 * q], b1), fmaf(wa, S.age[2 * q + 1], b1)) : pk2(b1, b1);
  }
  for (int w0 = 0; w0 < P.nwin; w0 += kWT) {
    const int nt = min(kWT, P.nwin - w0);
    for (int e = i; e < nt * kCh * kC; e += blockDim.x) {
      const int c = e % kC, r = e / kC;
      float a = 0.f, unused;
      if (state[c] == 1) window_max(P, S, w0 + r / kCh, r % kCh, c, -1, a, unused);
      S.d[r][c] = a;
    }
    __syncthreads();
    for (int wt = 0; wt < nt; ++wt) window_fma(P, S, wt, w0 + wt, h);
    __syncthreads();
  }
  const float dw3 = __ldg(P.w3 + (size_t)P.target * P.H + i) - __ldg(P.w3 + (size_t)(1 - P.target) * P.H + i);
  chain_probs(P, S, dw3, h);
  float prev = 0.f;
  if (i < kC) {
    prev = S.p[i];
    if (state[i]) P.p0[(size_t)(s0 + i) * P.G + g] = state[i] == 1 ? prev : NAN;
  }

  const int* perm = P.perm + g * P.K;
  for (int t = 0; t < P.K; ++t) {
    const int k = __ldg(perm + t);
    if (k < 0 || k >= P.K) {       // not a permutation entry: nothing is read, the chains' outputs become NaN
      if (i == 0) *P.bad = 1;
      if (i < kC) prev = NAN;
      continue;
    }
    const int wb = __ldg(P.win_ptr + k), we = __ldg(P.win_ptr + k + 1);
    for (int w0 = wb; w0 < we; w0 += kWT) {
      const int nt = min(kWT, we - w0);
      for (int e = i; e < nt * kCh * kC; e += blockDim.x) {
        const int c = e % kC, r = e / kC;
        float a = 0.f, b = 0.f;
        const int w = __ldg(P.win_idx + w0 + r / kCh);
        if (state[c] == 1 && w >= 0 && w < P.nwin) window_max(P, S, w, r % kCh, c, k, a, b);
        S.d[r][c] = b - a;
      }
      __syncthreads();
      for (int wt = 0; wt < nt; ++wt) {
        const int w = __ldg(P.win_idx + w0 + wt);
        if (w >= 0 && w < P.nwin) window_fma(P, S, wt, w, h);
      }
      __syncthreads();
    }
    if (i == 0) S.coal[k >> 5] |= 1u << (k & 31);    // seen by the next step after chain_probs' barriers
    chain_probs(P, S, dw3, h);
    if (i < kC && state[i]) {
      const float p = S.p[i];
      P.contrib[((size_t)(s0 + i) * P.G + g) * P.K + k] = state[i] == 1 ? p - prev : NAN;
      prev = p;
    }
  }
  if (i < kC && state[i]) P.pT[(size_t)(s0 + i) * P.G + g] = state[i] == 1 ? prev : NAN;
}

}  // namespace

extern "C" int mlg_shap_chains(const float* pat, int64_t n_pat, const float* bg, int64_t M, int64_t ld, int64_t Hg, int64_t Wg,
                               int64_t kh, int64_t kw, const float* w1p, const float* b1, const float* w1age, const float* age,
                               const float* w3, const float* b3, int target, int64_t H, const int32_t* owner,
                               const int32_t* win_ptr, const int32_t* win_idx, int64_t K, const int32_t* perm, int64_t G,
                               const int32_t* chain_pat, const int32_t* chain_bg, int64_t n_cp, float* contrib, float* p0,
                               float* pT, int32_t* bad, void* stream) {
  MLG_CHECK_ARG(pat && bg && w1p && b1 && w3 && b3 && owner && win_ptr && win_idx && perm && chain_pat && chain_bg && contrib &&
                    p0 && pT && bad && (!w1age || age),
                "mlg_shap_chains: null pointer");
  MLG_CHECK_ARG(n_pat >= 1 && M >= 1 && Hg >= 1 && Wg >= 1 && kh >= 1 && kw >= 1 && kh <= Hg && kw <= Wg &&
                    Hg * Wg <= kMaxCells && ld >= kCh * Hg * Wg,
                "mlg_shap_chains: bad grid sizes");
  MLG_CHECK_ARG(H >= 32 && H <= 512 && H % 32 == 0, "mlg_shap_chains: H must be a multiple of 32 in [32, 512] (got %lld)",
                (long long)H);
  MLG_CHECK_ARG(K >= 1 && K <= 32 * kMaxWords, "mlg_shap_chains: K must be in [1, %d]", 32 * kMaxWords);
  MLG_CHECK_ARG(target == 0 || target == 1, "mlg_shap_chains: target must be 0 or 1");
  MLG_CHECK_ARG(G >= 1 && n_cp >= 1, "mlg_shap_chains: no chain");
  const long long tiles = (n_cp + kC - 1) / kC;
  MLG_CHECK_ARG(tiles * G < (1ll << 31) && n_cp * G < (1ll << 40), "mlg_shap_chains: too many chains");
  ShapP P;
  memset(&P, 0, sizeof(P));
  P.pat = pat; P.bg = bg; P.ld = ld; P.n_pat = n_pat; P.M = M;
  P.Hg = (int)Hg; P.Wg = (int)Wg; P.kh = (int)kh; P.kw = (int)kw; P.Wo = (int)(Wg / kw);
  P.nwin = (int)((Hg / kh) * (Wg / kw)); P.cells = (int)(Hg * Wg);
  P.w1p = w1p; P.b1 = b1; P.w1age = w1age; P.age = w1age ? age : nullptr; P.w3 = w3; P.b3 = b3;
  P.target = target; P.H = (int)H;
  P.owner = owner; P.win_ptr = win_ptr; P.win_idx = win_idx; P.K = (int)K;
  P.perm = perm; P.G = G; P.n_cp = n_cp; P.chain_pat = chain_pat; P.chain_bg = chain_bg; P.tiles = (int)tiles;
  P.contrib = contrib; P.p0 = p0; P.pT = pT; P.bad = bad;
  const size_t smem = sizeof(Smem);
  MLG_CUDA(cudaFuncSetAttribute(shap_chains_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  shap_chains_kernel<<<(unsigned)(tiles * G), (unsigned)H, smem, (cudaStream_t)stream>>>(P);
  MLG_CHECK_LAUNCH("mlg_shap_chains");
  return MLG_OK;
}
