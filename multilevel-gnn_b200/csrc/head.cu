// MultilevelGNN's classification head and loss as FOUR kernels (two forward, two backward), sm_100a.
//
// Reference (models/multilevel_gnn.py:262-290, train.py:60,118): on the pooled pathway tensor [B, 32, 146, 3P]
//     Conv2d(32->32, 1x1) + ReLU, Conv2d(32->64, 1x1) + ReLU, MaxPool2d((kh, kw)), Dropout(0.25), flatten, cat(age),
//     Linear(F+1 -> D) + ReLU + Dropout(0.5), Linear(D -> 2), Softmax, BCELoss(weight [B,2]).
// As library ops that is ~60 launches per training step (each under 12 us: conv-as-GEMM x2, bias/ReLU, max-pool, two
// dropouts, cat, two Linears, softmax, BCE and all their backward ops) -- a fifth of the gbm step.  Here:
//   head_conv_pool_fwd   one warp per pooling window: both 1x1 convs of every pixel of the window as 32-lane mat-vecs
//                        (weights in shared memory, activations exchanged by shuffles), running max, dropout, and the
//                        result scattered straight into the flattened [B, F+1] matrix (age in the last column).
//   head_mlp_fwd         split-K batched GEMV over the [D, F+1] weight (the only real traffic: 7 MB for gbm), then one
//                        block per sample: bias + ReLU + dropout, Linear(D -> 2), softmax, weighted BCE, mean.
//   head_mlp_bwd         one pass over the [D, F+1] index space produces BOTH the weight gradient (written once) and
//                        the input gradient (the weight read once); the tiny softmax/BCE/Linear(D->2) backward is
//                        recomputed by every block.
//   head_conv_pool_bwd   recomputes the two convs per window (cheaper than saving 3 activations), routes the gradient to
//                        the first maximum (ATen's tie rule), back through both convs to the pooled features, and
//                        accumulates the four parameter gradients in registers; fixed-order two-level reduction.
// Dropout masks come from caller-provided random int32 words (torch's generator: graph-safe, torch.manual_seed applies);
// element kept iff bits >= p * 2^31.  Everything is fp32 FMA with fixed summation orders (deterministic).
#include <type_traits>

#include "common.cuh"
#include "../../include/mlg_b200.h"

namespace {

constexpr int CIN = 32, C1 = 32, C2 = 64;
constexpr int kWarps = 8;
constexpr int kThreads = kWarps * 32;
constexpr int kGradFloats = C1 * CIN + C1 + C2 * C1 + C2;   // gW1, gb1, gW2, gb2 = 3168

__device__ __forceinline__ bool drop_keep(const int* bits, size_t i, int thr) { return bits == nullptr || __ldg(bits + i) >= thr; }

// ---------------------------------------------------------------------------------------------------------------------
// conv 1x1 (32 -> 32) + ReLU, conv 1x1 (32 -> 64) + ReLU, max-pool, dropout, flatten.
// One THREAD per pixel: its 32 inputs, 32 hidden and 64 output values live in registers and every weight is read from
// shared memory as a warp-wide broadcast (LDS.128: four output channels per load), so the inner loops are pure FMA
// streams (1 LDS per 4 FMA).  A block owns whole "bands" (kh image rows = Wo pooling windows side by side), so pooling is
// a shared-memory exchange inside the block.  (The first version walked one warp per window with 32-lane shuffled
// mat-vecs: 28 us forward / 276 us backward on B200 -- shuffle / LDS bound; see profiles/r02_ncu_head.md.  Tried after this
// version and dropped: four threads per pixel in 64-pixel blocks, 576 blocks instead of 109 -- as adjacent lanes the
// weight reads stop being broadcasts (4 wavefronts per LDS.128: 31 / 68 us), as four warps per pixel group 27 / 54 us under
// ncu and the SAME step time in the captured graph, A/B on one box: 0.8276 vs 0.8271 ms.)
constexpr int kPix = 256;          // threads per block = pixel slots per block
constexpr int ZLD = C2 + 1;        // row pitch of the [pixel][64] tile: conflict-free for "thread = pixel" row access
constexpr int HLD = C1 + 4;        // row pitch of the [pixel][32] tiles (16-byte aligned rows)

struct ConvW {   // shared-memory weight copies; *t = [in][out] (forward), plain = [out][in] (backward)
  float w1t[CIN * C1];
  float w2t[C1 * C2];
  float w1[C1 * CIN];
  float w2[C2 * C1];
  float b1[C1];
  float b2[C2];
};

__device__ __forceinline__ void load_conv_weights(ConvW& S, const float* W1, const float* b1, const float* W2, const float* b2,
                                                  bool backward) {
  for (int t = threadIdx.x; t < C1 * CIN; t += blockDim.x) {
    const float v = __ldg(W1 + t);
    S.w1t[(t % CIN) * C1 + t / CIN] = v;
    if (backward) S.w1[t] = v;
  }
  for (int t = threadIdx.x; t < C2 * C1; t += blockDim.x) {
    const float v = __ldg(W2 + t);
    S.w2t[(t % C1) * C2 + t / C1] = v;
    if (backward) S.w2[t] = v;
  }
  for (int t = threadIdx.x; t < C1; t += blockDim.x) S.b1[t] = __ldg(b1 + t);
  for (int t = threadIdx.x; t < C2; t += blockDim.x) S.b2[t] = __ldg(b2 + t);
}

struct ConvPoolP {
  const float* x;   // [B, H, W, CIN] channel-last
  const float *W1, *b1, *W2, *b2;
  const float* age;   // [B] or NULL
  const int* bits;    // [B * F] or NULL
  int thr;            // keep iff bits >= thr
  float keep_scale;   // 1 / (1 - p)
  int B, H, W, kh, kw, Ho, Wo;
  int PB, NB, nbands;  // pixels per band (kh * W), bands per block, B * Ho
  int table;           // backward: per-(window, channel) argmax table in shared memory (kh * kw > 1)
  long long ld;       // row pitch of the flattened matrix
  float* a0;          // fwd out [B, ld]
  // backward
  const float* g_a0;  // [B, ld]
  float* g_x;         // [B, H, W, CIN]
  float* partial;     // [blocks, kGradFloats]
};

// this thread's pixel: returns false for idle slots.  band = (b, ho); p = dh * W + w inside the band.
__device__ __forceinline__ bool my_pixel(const ConvPoolP& P, int& bl, int& p, int& b, int& ho, size_t& pix) {
  bl = threadIdx.x / P.PB;
  p = threadIdx.x - bl * P.PB;
  const long long band = (long long)blockIdx.x * P.NB + bl;
  if (bl >= P.NB || band >= P.nbands) return false;
  b = (int)(band / P.Ho);
  ho = (int)(band - (long long)b * P.Ho);
  const int dh = p / P.W, w = p - dh * P.W;
  pix = ((size_t)b * P.H + (size_t)ho * P.kh + dh) * P.W + w;
  return true;
}

__device__ __forceinline__ void load_x(const float* x, size_t pix, float (&v)[CIN]) {
  const float4* src = reinterpret_cast<const float4*>(x + pix * CIN);
#pragma unroll
  for (int q = 0; q < CIN / 4; ++q) {
    const float4 t = __ldg(src + q);
    v[4 * q] = t.x; v[4 * q + 1] = t.y; v[4 * q + 2] = t.z; v[4 * q + 3] = t.w;
  }
}

// h1 = relu(W1 x + b1): weights broadcast from shared memory, four outputs per load
__device__ __forceinline__ void conv1(const ConvW& S, const float (&x)[CIN], float (&h)[C1]) {
#pragma unroll
  for (int j = 0; j < C1; ++j) h[j] = S.b1[j];
#pragma unroll
  for (int i = 0; i < CIN; ++i) {
#pragma unroll
    for (int j4 = 0; j4 < C1 / 4; ++j4) {
      const float4 w = *reinterpret_cast<const float4*>(&S.w1t[i * C1 + 4 * j4]);
      h[4 * j4] = fmaf(x[i], w.x, h[4 * j4]);
      h[4 * j4 + 1] = fmaf(x[i], w.y, h[4 * j4 + 1]);
      h[4 * j4 + 2] = fmaf(x[i], w.z, h[4 * j4 + 2]);
      h[4 * j4 + 3] = fmaf(x[i], w.w, h[4 * j4 + 3]);
    }
  }
#pragma unroll
  for (int j = 0; j < C1; ++j) h[j] = fmaxf(h[j], 0.f);
}

// relu(W2 h + b2) in four 16-channel chunks, written to this pixel's row of the [pixel][64] tile
__device__ __forceinline__ void conv2_to_tile(const ConvW& S, const float (&h)[C1], float* zrow) {
#pragma unroll
  for (int c0 = 0; c0 < C2; c0 += 16) {
    float a[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) a[c] = S.b2[c0 + c];
#pragma unroll
    for (int i = 0; i < C1; ++i) {
#pragma unroll
      for (int c4 = 0; c4 < 4; ++c4) {
        const float4 w = *reinterpret_cast<const float4*>(&S.w2t[i * C2 + c0 + 4 * c4]);
        a[4 * c4] = fmaf(h[i], w.x, a[4 * c4]);
        a[4 * c4 + 1] = fmaf(h[i], w.y, a[4 * c4 + 1]);
        a[4 * c4 + 2] = fmaf(h[i], w.z, a[4 * c4 + 2]);
        a[4 * c4 + 3] = fmaf(h[i], w.w, a[4 * c4 + 3]);
      }
    }
#pragma unroll
    for (int c = 0; c < 16; ++c) zrow[c0 + c] = fmaxf(a[c], 0.f);
  }
}

__global__ void __launch_bounds__(kPix) head_conv_pool_fwd_kernel(const ConvPoolP P) {
  extern __shared__ __align__(16) unsigned char head_smem[];
  ConvW& S = *reinterpret_cast<ConvW*>(head_smem);
  float* zt = reinterpret_cast<float*>(head_smem + sizeof(ConvW));   // [kPix][ZLD]
  load_conv_weights(S, P.W1, P.b1, P.W2, P.b2, false);
  __syncthreads();
  int bl, p, b, ho;
  size_t pix;
  if (my_pixel(P, bl, p, b, ho, pix)) {
    float x[CIN], h[C1];
    load_x(P.x, pix, x);
    conv1(S, x, h);
    conv2_to_tile(S, h, zt + threadIdx.x * ZLD);
  }
  __syncthreads();
  const long long HoWo = (long long)P.Ho * P.Wo, F = C2 * HoWo;
  for (int o = threadIdx.x; o < P.NB * P.Wo * C2; o += kPix) {
    const int c = o % C2, win = o / C2;
    const int wbl = win / P.Wo, wo = win - wbl * P.Wo;
    const long long band = (long long)blockIdx.x * P.NB + wbl;
    if (band >= P.nbands) break;
    const int bb = (int)(band / P.Ho), hho = (int)(band - (long long)bb * P.Ho);
    float best = 0.f;    // post-ReLU values are >= 0
    for (int dh = 0; dh < P.kh; ++dh)
      for (int dw = 0; dw < P.kw; ++dw) best = fmaxf(best, zt[(wbl * P.PB + dh * P.W + wo * P.kw + dw) * ZLD + c]);
    const size_t col = (size_t)c * HoWo + (size_t)hho * P.Wo + wo;
    P.a0[(size_t)bb * P.ld + col] = drop_keep(P.bits, (size_t)bb * F + col, P.thr) ? best * P.keep_scale : 0.f;
    if (P.age && c == 0 && hho == 0 && wo == 0) P.a0[(size_t)bb * P.ld + F] = __ldg(P.age + bb);
  }
}

__global__ void __launch_bounds__(kPix) head_conv_pool_bwd_kernel(const ConvPoolP P) {
  extern __shared__ __align__(16) unsigned char head_smem[];
  ConvW& S = *reinterpret_cast<ConvW*>(head_smem);
  float* zt = reinterpret_cast<float*>(head_smem + sizeof(ConvW));   // [kPix][ZLD]: relu(z2), then dL/dz2
  float* Ht = zt + kPix * ZLD;                                        // [kPix][HLD]: h1
  float* Xt = Ht + kPix * HLD;                                        // [kPix][HLD]: x
  float* G1 = Xt + kPix * HLD;                                        // [kPix][HLD]: dL/dz1
  float* gval = G1 + kPix * HLD;                                      // [NB * Wo][64]: gradient reaching each window maximum
  unsigned char* garg = reinterpret_cast<unsigned char*>(gval + P.NB * P.Wo * C2);   // its window position (255: none)
  load_conv_weights(S, P.W1, P.b1, P.W2, P.b2, true);
  __syncthreads();
  int bl = 0, p = 0, b = 0, ho = 0;
  size_t pix = 0;
  const bool live = my_pixel(P, bl, p, b, ho, pix);
  float h[C1];
  {
    float x[CIN];
    if (live) {
      load_x(P.x, pix, x);
      conv1(S, x, h);
      conv2_to_tile(S, h, zt + threadIdx.x * ZLD);
    } else {
#pragma unroll
      for (int i = 0; i < CIN; ++i) x[i] = 0.f;
#pragma unroll
      for (int i = 0; i < C1; ++i) h[i] = 0.f;
      for (int c = 0; c < C2; ++c) zt[threadIdx.x * ZLD + c] = 0.f;
    }
#pragma unroll
    for (int i = 0; i < CIN; ++i) Xt[threadIdx.x * HLD + i] = x[i];
#pragma unroll
    for (int i = 0; i < C1; ++i) Ht[threadIdx.x * HLD + i] = h[i];
  }
  __syncthreads();
  // gradient routed to the FIRST maximum of every (window, channel); nothing where the maximum is the clamped 0
  const long long HoWo = (long long)P.Ho * P.Wo, F = C2 * HoWo;
  for (int o = threadIdx.x; o < (P.table ? P.NB * P.Wo * C2 : 0); o += kPix) {
    const int c = o % C2, win = o / C2;
    const int wbl = win / P.Wo, wo = win - wbl * P.Wo;
    const long long band = (long long)blockIdx.x * P.NB + wbl;
    float g = 0.f;
    int arg = 255;
    if (band < P.nbands) {
      const int bb = (int)(band / P.Ho), hho = (int)(band - (long long)bb * P.Ho);
      float best = 0.f;
      for (int dh = 0; dh < P.kh; ++dh)
        for (int dw = 0; dw < P.kw; ++dw) {
          const float v = zt[(wbl * P.PB + dh * P.W + wo * P.kw + dw) * ZLD + c];
          if (v > best) { best = v; arg = dh * P.W + wo * P.kw + dw; }     // position inside the band
        }
      if (arg != 255) {
        const size_t col = (size_t)c * HoWo + (size_t)hho * P.Wo + wo;
        g = drop_keep(P.bits, (size_t)bb * F + col, P.thr) ? __ldg(P.g_a0 + (size_t)bb * P.ld + col) * P.keep_scale : 0.f;
      }
    }
    gval[o] = g;
    garg[o] = (unsigned char)arg;
  }
  __syncthreads();
  // per pixel: dL/dz2 (into the tile), back through conv2 / ReLU / conv1
  {
    float gh[C1];
#pragma unroll
    for (int i = 0; i < C1; ++i) gh[i] = 0.f;
    const int dh = p / P.W, w = p - dh * P.W;
    const int wo = w / P.kw;
    const bool in_window = live && wo < P.Wo;
    float* zrow = zt + threadIdx.x * ZLD;
    for (int c = 0; c < C2; ++c) {
      float gz = 0.f;
      if (in_window) {
        if (P.table) {
          const int o = (bl * P.Wo + wo) * C2 + c;
          gz = (int)garg[o] == p ? gval[o] : 0.f;
        } else if (zrow[c] > 0.f) {        // 1 x 1 windows: every pixel is its own maximum
          const size_t col = (size_t)c * HoWo + (size_t)ho * P.Wo + wo;
          gz = drop_keep(P.bits, (size_t)b * F + col, P.thr) ? __ldg(P.g_a0 + (size_t)b * P.ld + col) * P.keep_scale : 0.f;
        }
      }
      zrow[c] = gz;
      if (gz != 0.f) {
#pragma unroll
        for (int i4 = 0; i4 < C1 / 4; ++i4) {
          const float4 wv = *reinterpret_cast<const float4*>(&S.w2[c * C1 + 4 * i4]);
          gh[4 * i4] = fmaf(gz, wv.x, gh[4 * i4]);
          gh[4 * i4 + 1] = fmaf(gz, wv.y, gh[4 * i4 + 1]);
          gh[4 * i4 + 2] = fmaf(gz, wv.z, gh[4 * i4 + 2]);
          gh[4 * i4 + 3] = fmaf(gz, wv.w, gh[4 * i4 + 3]);
        }
      }
    }
    float gx[CIN];
#pragma unroll
    for (int i = 0; i < CIN; ++i) gx[i] = 0.f;
#pragma unroll
    for (int j = 0; j < C1; ++j) {
      const float gz1 = h[j] > 0.f ? gh[j] : 0.f;
      G1[threadIdx.x * HLD + j] = gz1;
#pragma unroll
      for (int i4 = 0; i4 < CIN / 4; ++i4) {
        const float4 wv = *reinterpret_cast<const float4*>(&S.w1[j * CIN + 4 * i4]);
        gx[4 * i4] = fmaf(gz1, wv.x, gx[4 * i4]);
        gx[4 * i4 + 1] = fmaf(gz1, wv.y, gx[4 * i4 + 1]);
        gx[4 * i4 + 2] = fmaf(gz1, wv.z, gx[4 * i4 + 2]);
        gx[4 * i4 + 3] = fmaf(gz1, wv.w, gx[4 * i4 + 3]);
      }
    }
    if (live) {
      float4* dst = reinterpret_cast<float4*>(P.g_x + pix * CIN);
#pragma unroll
      for (int q = 0; q < CIN / 4; ++q) dst[q] = make_float4(gx[4 * q], gx[4 * q + 1], gx[4 * q + 2], gx[4 * q + 3]);
    }
  }
  if (!P.partial) return;   // input gradient only
  __syncthreads();
  // parameter gradients of this block: gW2 = Gz2^T H1 (64 x 32), gW1 = Gz1^T X (32 x 32), column sums; fixed order over pixels
  float* part = P.partial + (size_t)blockIdx.x * kGradFloats;
  {
    const int c = threadIdx.x >> 2, i0 = (threadIdx.x & 3) * 8;      // 64 x (4 x 8)
    float acc[8], sb = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) acc[q] = 0.f;
    for (int t = 0; t < kPix; ++t) {
      const float g = zt[t * ZLD + c];
      const float4 h0 = *reinterpret_cast<const float4*>(&Ht[t * HLD + i0]);
      const float4 h1v = *reinterpret_cast<const float4*>(&Ht[t * HLD + i0 + 4]);
      acc[0] = fmaf(g, h0.x, acc[0]); acc[1] = fmaf(g, h0.y, acc[1]); acc[2] = fmaf(g, h0.z, acc[2]); acc[3] = fmaf(g, h0.w, acc[3]);
      acc[4] = fmaf(g, h1v.x, acc[4]); acc[5] = fmaf(g, h1v.y, acc[5]); acc[6] = fmaf(g, h1v.z, acc[6]); acc[7] = fmaf(g, h1v.w, acc[7]);
      sb += g;
    }
    float* gw2 = part + C1 * CIN + C1;
#pragma unroll
    for (int q = 0; q < 8; ++q) gw2[c * C1 + i0 + q] = acc[q];
    if ((threadIdx.x & 3) == 0) gw2[C2 * C1 + c] = sb;
  }
  {
    const int j = threadIdx.x >> 3, i0 = (threadIdx.x & 7) * 4;      // 32 x (8 x 4)
    float acc[4] = {0.f, 0.f, 0.f, 0.f}, sb = 0.f;
    for (int t = 0; t < kPix; ++t) {
      const float g = G1[t * HLD + j];
      const float4 xv = *reinterpret_cast<const float4*>(&Xt[t * HLD + i0]);
      acc[0] = fmaf(g, xv.x, acc[0]); acc[1] = fmaf(g, xv.y, acc[1]); acc[2] = fmaf(g, xv.z, acc[2]); acc[3] = fmaf(g, xv.w, acc[3]);
      sb += g;
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) part[j * CIN + i0 + q] = acc[q];
    if ((threadIdx.x & 7) == 0) part[C1 * CIN + j] = sb;
  }
}

// zero gradient for the image rows the floor-mode pool never reads (pixels of whole tail rows; tail COLUMNS are written
// by the band threads above)
__global__ void head_conv_tail_zero_kernel(float4* __restrict__ g_x, int B, int H, int W, int row0) {
  const long long per_b = (long long)(H - row0) * W * (CIN / 4);
  const long long total = per_b * B;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long b = i / per_b, r = i - b * per_b;
    g_x[((size_t)b * H + row0) * W * (CIN / 4) + r] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

__global__ void head_conv_reduce_kernel(const float* __restrict__ partial, int nblocks, float* __restrict__ gW1,
                                        float* __restrict__ gb1, float* __restrict__ gW2, float* __restrict__ gb2) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= kGradFloats) return;
  float s = 0.f;
  for (int b = 0; b < nblocks; ++b) s += partial[(size_t)b * kGradFloats + t];
  if (t < C1 * CIN) gW1[t] = s;
  else if (t < C1 * CIN + C1) gb1[t - C1 * CIN] = s;
  else if (t < C1 * CIN + C1 + C2 * C1) gW2[t - C1 * CIN - C1] = s;
  else gb2[t - C1 * CIN - C1 - C2 * C1] = s;
}

// geometry shared by both directions: bands per block and grid size; false when a band does not fit one block
inline size_t conv_pool_smem(const ConvPoolP& P, bool backward) {
  size_t s = sizeof(ConvW) + (size_t)kPix * ZLD * 4;
  if (backward) s += 3 * (size_t)kPix * HLD * 4 + (P.table ? (size_t)P.NB * P.Wo * C2 * 5 : 0) + 16;
  return s;
}
inline bool conv_pool_geometry(ConvPoolP& P) {
  P.PB = P.kh * P.W;
  if (P.PB > kPix || P.PB > 255) return false;
  P.NB = kPix / P.PB;
  P.nbands = P.B * P.Ho;
  P.table = (P.kh * P.kw > 1) ? 1 : 0;
  while (P.NB > 1 && conv_pool_smem(P, true) > 227 * 1024) --P.NB;     // the argmax table of many small windows
  return true;
}
inline int conv_pool_blocks(const ConvPoolP& P) { return (P.nbands + P.NB - 1) / P.NB; }

// ------------------------------------------------------------------------------------------------------------
// MLP + loss
// ------------------------------------------------------------------------------------------------------------
// One block = one 64-column slice of K, one thread = one hidden unit n (blockDim = D): the slice of W0 [D x 64] and of
// a0 [R x 64] (transposed) are staged in shared memory once; every thread then owns acc[r] for all R samples and streams
// its W row against broadcast a0 values (LDS.128: four samples per load).  The backward kernel has the same geometry and
// produces, from ONE staged W slice, both the slice of the weight gradient and the slice of the input gradient.
// K columns per block: 64, or 32 when 64 samples x 512 hidden units would not fit shared memory next to a 64-wide slice
// (row pitch of the staged W slice = KSL + 1: "thread = row" access is conflict-free)

struct MlpP {
  const float* a0;   // [R, ld_a] (K columns used)
  const float* W0;   // [D, K] row pitch K
  const float* b0;   // [D]
  const float* W3;   // [2, D]
  const float* b3;   // [2]
  const int* bits;   // [R * D] or NULL
  int thr;
  float keep_scale;
  const float* y;        // [R, 2] or NULL (no loss)
  const float* weight;   // [R, 2] or NULL
  int R, D, K, slices;
  long long ld_a;
  float* partial;   // [slices, R, D]
  float* a1;        // [R, D] post ReLU + dropout
  float* pred;      // [R, 2]
  float* rowloss;   // [R]
  float* loss;      // [1]
  unsigned* counter;
};

// stage W0[:, k0 : k0 + 64] as Ws[n][k] and a0[:, k0 : k0 + 64] as As[k][r] (zero padded past K / R)
template <int RT, int KSL>
__device__ __forceinline__ void stage_slices(const float* W0, int D, int K, const float* a0, long long ld_a, int R, int k0,
                                             float* Ws, float* As) {
  constexpr int WLD = KSL + 1;
  constexpr int RU = 8;     // rows whose loads are in flight together (r02 ncu: one row at a time = 25 us of pure latency)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  for (int n0 = warp; n0 < D; n0 += nwarps * RU) {
    float v[RU][KSL / 32];
#pragma unroll
    for (int u = 0; u < RU; ++u) {
      const int n = n0 + u * nwarps;
      const float* row = W0 + (size_t)(n < D ? n : 0) * K + k0;
#pragma unroll
      for (int q = 0; q < KSL / 32; ++q) v[u][q] = (n < D && k0 + lane + 32 * q < K) ? __ldg(row + lane + 32 * q) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < RU; ++u) {
      const int n = n0 + u * nwarps;
      if (n < D) {
#pragma unroll
        for (int q = 0; q < KSL / 32; ++q) Ws[n * WLD + lane + 32 * q] = v[u][q];
      }
    }
  }
  // a0 slice transposed to [k][r]: thread -> (k = t % KSL, rows r = t / KSL, + step), loads batched like above
  const int kk = threadIdx.x % KSL, rstep = blockDim.x / KSL;
  {
    float v[RT / 4];     // blockDim >= 4 * KSL  =>  rstep >= 4  =>  at most RT / 4 rows per thread
    const int rfirst = threadIdx.x / KSL;
#pragma unroll
    for (int c = 0; c < RT / 4; ++c) {
      const int r = rfirst + c * rstep;
      v[c] = (r < R && k0 + kk < K) ? __ldg(a0 + (size_t)r * ld_a + k0 + kk) : 0.f;
    }
#pragma unroll
    for (int c = 0; c < RT / 4; ++c) {
      const int r = rfirst + c * rstep;
      if (r < RT) As[kk * RT + r] = v[c];
    }
  }
}

// Forward partial products.  Block = (32 hidden units) x (one K group of KG = 512 columns); thread = (unit n = lane,
// sub-slice g = warp of 64 columns): acc[r] over its 64 columns for all samples, then the 8 sub-slices are added in a fixed
// order through shared memory -> ONE partial per (K group, sample, unit): 14 partial slices for K = 6913 instead of 109
// (the finish kernel then has 14 loads per output instead of 109: r02 ncu 49 us -> see profiles/r02_ncu_head.md).
constexpr int KG = 512, KSUB = 64, NG = 32;
constexpr int WG_LD = KG + 1;

template <int RT>
__global__ void __launch_bounds__(256) head_mlp_partial_kernel(const MlpP P) {
  extern __shared__ __align__(16) float mlp_sm[];
  float* Ws = mlp_sm;                   // [NG][WG_LD]
  float* As = Ws + NG * WG_LD;          // [KG][RT]; afterwards the [8][RT][NG] reduction buffer
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n0 = blockIdx.x * NG, k0 = blockIdx.y * KG;
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) *P.counter = 0u;   // the finish kernel's arrival counter
  // stage W0[n0 : n0 + 32, k0 : k0 + 512] (each row: 2 KB contiguous) -- four rows' loads in flight per warp step
  for (int rr = warp; rr < NG; rr += 8 * 4) {
    float v[4][KG / 32];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int n = n0 + rr + 8 * u;
      const float* row = P.W0 + (size_t)(n < P.D ? n : 0) * P.K + k0;
#pragma unroll
      for (int q = 0; q < KG / 32; ++q) v[u][q] = (n < P.D && k0 + lane + 32 * q < P.K) ? __ldg(row + lane + 32 * q) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int q = 0; q < KG / 32; ++q) Ws[(rr + 8 * u) * WG_LD + lane + 32 * q] = v[u][q];
  }
  // a0[:, k0 : k0 + 512] transposed to As[k][r]: thread -> column k = tid (+256), RT loads in flight
#pragma unroll
  for (int half = 0; half < KG / 256; ++half) {
    const int k = threadIdx.x + 256 * half;
    float v[RT];
#pragma unroll
    for (int r = 0; r < RT; ++r) v[r] = (r < P.R && k0 + k < P.K) ? __ldg(P.a0 + (size_t)r * P.ld_a + k0 + k) : 0.f;
#pragma unroll
    for (int r4 = 0; r4 < RT / 4; ++r4)
      *reinterpret_cast<float4*>(&As[k * RT + 4 * r4]) = make_float4(v[4 * r4], v[4 * r4 + 1], v[4 * r4 + 2], v[4 * r4 + 3]);
  }
  __syncthreads();
  float acc[RT];
#pragma unroll
  for (int r = 0; r < RT; ++r) acc[r] = 0.f;
  const float* wrow = Ws + lane * WG_LD + warp * KSUB;
  const float* arow = As + (size_t)warp * KSUB * RT;
#pragma unroll 4
  for (int k = 0; k < KSUB; ++k) {
    const float w = wrow[k];
#pragma unroll
    for (int r4 = 0; r4 < RT / 4; ++r4) {
      const float4 a = *reinterpret_cast<const float4*>(&arow[k * RT + 4 * r4]);
      acc[4 * r4] = fmaf(w, a.x, acc[4 * r4]);
      acc[4 * r4 + 1] = fmaf(w, a.y, acc[4 * r4 + 1]);
      acc[4 * r4 + 2] = fmaf(w, a.z, acc[4 * r4 + 2]);
      acc[4 * r4 + 3] = fmaf(w, a.w, acc[4 * r4 + 3]);
    }
  }
  __syncthreads();                       // As is dead: reuse it as [8 sub-slices][RT][NG]
  float* red = As;
#pragma unroll
  for (int r = 0; r < RT; ++r) red[(warp * RT + r) * NG + lane] = acc[r];
  __syncthreads();
  for (int t = threadIdx.x; t < RT * NG; t += 256) {
    const int r = t / NG, l = t - r * NG;
    if (r < P.R && n0 + l < P.D) {
      float s = 0.f;
#pragma unroll
      for (int g = 0; g < 8; ++g) s += red[(g * RT + r) * NG + l];
      P.partial[((size_t)blockIdx.y * P.R + r) * P.D + n0 + l] = s;
    }
  }
}

// one block per sample r: slice reduction + bias + ReLU + dropout -> a1[r, :]; logits, softmax, weighted BCE; the last
// block to finish sums the per-sample losses in index order
__global__ void __launch_bounds__(kThreads) head_mlp_finish_kernel(const MlpP P) {
  __shared__ float red[2][kWarps];
  __shared__ int is_last;
  const int r = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float z0 = 0.f, z1 = 0.f;
  for (int n = threadIdx.x; n < P.D; n += kThreads) {
    // eight loads in flight, eight independent chains combined in a fixed order
    float c8[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) c8[q] = 0.f;
    const float* pp = P.partial + (size_t)r * P.D + n;
    const size_t st = (size_t)P.R * P.D;
    int g = 0;
    for (; g + 8 <= P.slices; g += 8) {
      float v[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) v[q] = pp[(size_t)(g + q) * st];
#pragma unroll
      for (int q = 0; q < 8; ++q) c8[q] += v[q];
    }
    for (; g < P.slices; ++g) c8[0] += pp[(size_t)g * st];
    float s = ((c8[0] + c8[1]) + (c8[2] + c8[3])) + ((c8[4] + c8[5]) + (c8[6] + c8[7]));
    s += __ldg(P.b0 + n);
    s = fmaxf(s, 0.f);
    s = drop_keep(P.bits, (size_t)r * P.D + n, P.thr) ? s * P.keep_scale : 0.f;
    P.a1[(size_t)r * P.D + n] = s;
    z0 = fmaf(s, __ldg(P.W3 + n), z0);
    z1 = fmaf(s, __ldg(P.W3 + P.D + n), z1);
  }
  z0 = warp_sum(z0);
  z1 = warp_sum(z1);
  if (lane == 0) { red[0][warp] = z0; red[1][warp] = z1; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = __ldg(P.b3), b = __ldg(P.b3 + 1);
    for (int w = 0; w < kWarps; ++w) { a += red[0][w]; b += red[1][w]; }
    const float m = fmaxf(a, b);
    const float ea = expf(a - m), eb = expf(b - m);
    const float inv = 1.f / (ea + eb);
    const float p0 = ea * inv, p1 = eb * inv;
    P.pred[2 * r] = p0;
    P.pred[2 * r + 1] = p1;
    if (P.y) {
      // BCELoss: -(y log p + (1 - y) log(1 - p)), logs clamped at -100 (ATen), times weight
      const float y0 = __ldg(P.y + 2 * r), y1 = __ldg(P.y + 2 * r + 1);
      const float w0 = P.weight ? __ldg(P.weight + 2 * r) : 1.f, w1 = P.weight ? __ldg(P.weight + 2 * r + 1) : 1.f;
      const float l0 = -(y0 * fmaxf(logf(p0), -100.f) + (1.f - y0) * fmaxf(logf(1.f - p0), -100.f)) * w0;
      const float l1 = -(y1 * fmaxf(logf(p1), -100.f) + (1.f - y1) * fmaxf(logf(1.f - p1), -100.f)) * w1;
      P.rowloss[r] = l0 + l1;
      __threadfence();
      const unsigned c = atomicAdd(P.counter, 1u);
      is_last = (c == gridDim.x - 1);
    } else {
      is_last = 0;
    }
  }
  __syncthreads();
  if (is_last && threadIdx.x == 0) {
    __threadfence();
    float s = 0.f;
    for (int i = 0; i < P.R; ++i) s += *reinterpret_cast<volatile float*>(P.rowloss + i);
    P.loss[0] = s / (2.f * (float)P.R);
    *P.counter = 0u;
  }
}

struct MlpBwdP {
  const float* g_pred;   // [R, 2] or NULL
  const float* g_loss;   // [1] or NULL
  const float *pred, *y, *weight;
  const float *a0, *a1, *W0, *W3;
  int R, D, K;
  long long ld_a, ld_g;
  float keep_scale;
  float *g_a0, *g_W0, *g_b0, *g_W3, *g_b3;
};

// Rows of dL/dz1 per thread group in head_mlp_bwd_kernel's input-gradient pass: the smallest of 4, 8, 16 whose ngrp groups
// cover all RT rows.  RT (32 or 64) is a multiple of each choice, so a group that starts below RT also ends at or below it:
// no group reads past the RT x D dL/dz1 tile, and none is skipped.  A plain ceil(RT / ngrp) gives 5, 6 or 7 for
// D in 320..480, which the unrolled loop cannot take.
__host__ __device__ inline int mlp_bwd_rows_per_group(int RT, int ngrp) {
  const int need = (RT + ngrp - 1) / ngrp;
  return need <= 4 ? 4 : need <= 8 ? 8 : 16;
}

template <int RT, int KSL>
__global__ void __launch_bounds__(512) head_mlp_bwd_kernel(const MlpBwdP P) {
  constexpr int KS = KSL, WLD = KSL + 1;
  extern __shared__ __align__(16) float mlp_sm[];
  float* Ws = mlp_sm;                   // [D][WLD]: W0 slice, later the gW0 slice
  float* As = Ws + P.D * WLD;           // [KS][RT]
  float* Gs = As + KS * RT;             // [RT][D]: dL/dz1
  float* gz2 = Gs + RT * P.D;           // [RT][2]
  const int n = threadIdx.x, k0 = blockIdx.x * KS, D = P.D;
  stage_slices<RT, KSL>(P.W0, D, P.K, P.a0, P.ld_a, P.R, k0, Ws, As);
  // ---- softmax + BCE backward -> dL/dlogits (every block recomputes these R x 2 values) ----
  for (int r = threadIdx.x; r < RT; r += blockDim.x) {
    float o0 = 0.f, o1 = 0.f;
    if (r < P.R) {
      const float p0 = __ldg(P.pred + 2 * r), p1 = __ldg(P.pred + 2 * r + 1);
      float g0 = P.g_pred ? __ldg(P.g_pred + 2 * r) : 0.f, g1 = P.g_pred ? __ldg(P.g_pred + 2 * r + 1) : 0.f;
      if (P.g_loss && P.y) {
        const float gl = __ldg(P.g_loss) / (2.f * (float)P.R);
        const float y0 = __ldg(P.y + 2 * r), y1 = __ldg(P.y + 2 * r + 1);
        const float w0 = P.weight ? __ldg(P.weight + 2 * r) : 1.f, w1 = P.weight ? __ldg(P.weight + 2 * r + 1) : 1.f;
        // ATen binary_cross_entropy_backward: (p - y) / max((1 - p) p, 1e-12) * weight
        g0 += gl * w0 * (p0 - y0) / fmaxf((1.f - p0) * p0, 1e-12f);
        g1 += gl * w1 * (p1 - y1) / fmaxf((1.f - p1) * p1, 1e-12f);
      }
      const float dot = g0 * p0 + g1 * p1;
      o0 = p0 * (g0 - dot);
      o1 = p1 * (g1 - dot);
    }
    gz2[2 * r] = o0;
    gz2[2 * r + 1] = o1;
  }
  __syncthreads();
  // ---- this thread's hidden unit: dL/dz1[r][n] for every sample, in registers and in shared memory ----
  float gz[RT];
  const bool unit = n < D;      // helper threads of a narrow layer (blockDim = max(D, 256)) own no hidden unit
#pragma unroll
  for (int r = 0; r < RT; ++r) gz[r] = 0.f;
  if (unit) {
    const float w30 = __ldg(P.W3 + n), w31 = __ldg(P.W3 + D + n);
    float a1v[RT];
#pragma unroll
    for (int r = 0; r < RT; ++r) a1v[r] = r < P.R ? __ldg(P.a1 + (size_t)r * D + n) : 0.f;
#pragma unroll
    for (int r = 0; r < RT; ++r) {
      gz[r] = a1v[r] > 0.f ? (gz2[2 * r] * w30 + gz2[2 * r + 1] * w31) * P.keep_scale : 0.f;
      Gs[r * D + n] = gz[r];
    }
    if (blockIdx.x == 0 && P.g_W0) {   // the small parameter gradients, fixed order over the samples
      float s = 0.f, u0 = 0.f, u1 = 0.f;
#pragma unroll
      for (int r = 0; r < RT; ++r) {
        s += gz[r];
        u0 = fmaf(gz2[2 * r], a1v[r], u0);
        u1 = fmaf(gz2[2 * r + 1], a1v[r], u1);
      }
      P.g_b0[n] = s;
      P.g_W3[n] = u0;
      P.g_W3[D + n] = u1;
      if (n < 2) {
        float t = 0.f;
        for (int r = 0; r < P.R; ++r) t += gz2[2 * r + n];
        P.g_b3[n] = t;
      }
    }
  }
  __syncthreads();
  // ---- input gradient slice: g_a0[r][k0 + k] = sum_n dz1[r][n] W0[n][k0 + k]; thread = (k, group of rows) ----
  if (P.g_a0) {
    const int k = threadIdx.x & (KS - 1), grp = threadIdx.x / KS, ngrp = blockDim.x / KS;
    const int rpg = mlp_bwd_rows_per_group(RT, ngrp);
    const int r0 = grp * rpg;
    float acc[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) acc[q] = 0.f;
    auto run = [&](auto rpg_c) {
      constexpr int RPG = decltype(rpg_c)::value;
      const float* gp = Gs + (size_t)(r0 < RT ? r0 : 0) * D;
      for (int nn = 0; nn < D; nn += 4) {
        const float w0 = Ws[nn * WLD + k], w1 = Ws[(nn + 1) * WLD + k], w2 = Ws[(nn + 2) * WLD + k], w3 = Ws[(nn + 3) * WLD + k];
#pragma unroll
        for (int q = 0; q < RPG; ++q) {
          const float4 g4 = *reinterpret_cast<const float4*>(gp + (size_t)q * D + nn);
          acc[q] = fmaf(g4.x, w0, fmaf(g4.y, w1, fmaf(g4.z, w2, fmaf(g4.w, w3, acc[q]))));
        }
      }
    };
    if (r0 + rpg <= RT) {
      if (rpg == 4) run(std::integral_constant<int, 4>());
      else if (rpg == 8) run(std::integral_constant<int, 8>());
      else run(std::integral_constant<int, 16>());
    }
    if (k0 + k < P.K) {
#pragma unroll
      for (int q = 0; q < 16; ++q)
        if (q < rpg && r0 + q < P.R) P.g_a0[(size_t)(r0 + q) * P.ld_g + k0 + k] = acc[q];
    }
  }
  if (!P.g_W0) return;   // input gradient only
  __syncthreads();
  // ---- weight gradient slice: gW0[n][k0 + k] = sum_r dz1[r][n] a0[r][k0 + k]; staged in Ws, then written row by row ----
  if (unit) {
#pragma unroll 4
    for (int k = 0; k < KS; ++k) {
      float v = 0.f;
#pragma unroll
      for (int r4 = 0; r4 < RT / 4; ++r4) {
        const float4 a = *reinterpret_cast<const float4*>(&As[k * RT + 4 * r4]);
        v = fmaf(gz[4 * r4], a.x, v);
        v = fmaf(gz[4 * r4 + 1], a.y, v);
        v = fmaf(gz[4 * r4 + 2], a.z, v);
        v = fmaf(gz[4 * r4 + 3], a.w, v);
      }
      Ws[n * WLD + k] = v;
    }
  }
  __syncthreads();
  {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    for (int row = warp; row < D; row += nwarps) {
      float* dst = P.g_W0 + (size_t)row * P.K + k0;
#pragma unroll
      for (int q = 0; q < KS; q += 32)
        if (k0 + lane + q < P.K) dst[lane + q] = Ws[row * WLD + lane + q];
    }
  }
}

// K columns per block (see head_mlp_*_kernel) and the resulting number of K slices; one choice for forward and backward
inline int mlp_ks(int64_t R, int64_t D) { return (R > 32 && D > 256) ? 32 : 64; }
inline int mlp_slices(int64_t R, int64_t D, int64_t K) { const int ks = mlp_ks(R, D); return (int)((K + ks - 1) / ks); }   // backward
inline int mlp_fwd_slices(int64_t K) { return (int)((K + KG - 1) / KG); }

inline int drop_threshold(float p) {
  if (!(p > 0.f)) return 0;
  double t = (double)p * 2147483648.0;
  if (t > 2147483647.0) t = 2147483647.0;
  return (int)t;
}

}  // namespace

extern "C" int mlg_head_conv_pool_supported(int64_t cin, int64_t c1, int64_t c2) { return cin == CIN && c1 == C1 && c2 == C2; }

static int conv_pool_fill(ConvPoolP& P, const float* x_cl, const float* W1, const float* b1, const float* W2, const float* b2,
                          const int32_t* drop_bits, float drop_p, int64_t B, int64_t H, int64_t W, int64_t kh, int64_t kw) {
  memset(&P, 0, sizeof(P));
  P.x = x_cl; P.W1 = W1; P.b1 = b1; P.W2 = W2; P.b2 = b2;
  P.bits = drop_p > 0.f ? drop_bits : nullptr;
  P.thr = drop_threshold(drop_p); P.keep_scale = 1.f / (1.f - drop_p);
  P.B = (int)B; P.H = (int)H; P.W = (int)W; P.kh = (int)kh; P.kw = (int)kw; P.Ho = (int)(H / kh); P.Wo = (int)(W / kw);
  MLG_CHECK_ARG(conv_pool_geometry(P), "mlg_head_conv_pool: one band (kh * W = %lld pixels) must fit a 255-pixel block", (long long)(kh * W));
  MLG_CHECK_ARG((uintptr_t)x_cl % 16 == 0, "mlg_head_conv_pool: x_cl must be 16-byte aligned");
  return MLG_OK;
}

extern "C" int64_t mlg_head_conv_pool_bwd_workspace_bytes(int64_t B, int64_t H, int64_t W, int64_t kh, int64_t kw) {
  if (kh < 1 || kw < 1 || kh * W > 255) return 0;
  ConvPoolP P;
  memset(&P, 0, sizeof(P));
  P.B = (int)B; P.H = (int)H; P.W = (int)W; P.kh = (int)kh; P.kw = (int)kw; P.Ho = (int)(H / kh); P.Wo = (int)(W / kw);
  conv_pool_geometry(P);
  return (int64_t)conv_pool_blocks(P) * kGradFloats * 4;
}

extern "C" int mlg_head_conv_pool_fwd(const float* x_cl, const float* W1, const float* b1, const float* W2, const float* b2,
                                      const float* age, const int32_t* drop_bits, float drop_p, int64_t B, int64_t H,
                                      int64_t W, int64_t kh, int64_t kw, float* a0, int64_t ld, void* stream) {
  MLG_CHECK_ARG(x_cl && W1 && b1 && W2 && b2 && a0, "mlg_head_conv_pool_fwd: null pointer");
  MLG_CHECK_ARG(B >= 1 && H >= 1 && W >= 1 && kh >= 1 && kw >= 1 && kh <= H && kw <= W, "mlg_head_conv_pool_fwd: bad sizes");
  MLG_CHECK_ARG(drop_p >= 0.f && drop_p < 1.f, "mlg_head_conv_pool_fwd: dropout p must be in [0, 1)");
  MLG_CHECK_ARG(drop_p == 0.f || drop_bits, "mlg_head_conv_pool_fwd: dropout needs drop_bits");
  ConvPoolP P;
  if (int rc = conv_pool_fill(P, x_cl, W1, b1, W2, b2, drop_bits, drop_p, B, H, W, kh, kw)) return rc;
  P.age = age;
  const long long F = (long long)C2 * P.Ho * P.Wo;
  MLG_CHECK_ARG(ld >= F + (age ? 1 : 0), "mlg_head_conv_pool_fwd: ld too small");
  P.ld = ld; P.a0 = a0;
  const size_t smem = conv_pool_smem(P, false);
  MLG_CUDA(cudaFuncSetAttribute(head_conv_pool_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  head_conv_pool_fwd_kernel<<<conv_pool_blocks(P), kPix, smem, (cudaStream_t)stream>>>(P);
  MLG_CHECK_LAUNCH("mlg_head_conv_pool_fwd");
  return MLG_OK;
}

extern "C" int mlg_head_conv_pool_bwd(const float* g_a0, int64_t ld, const float* x_cl, const float* W1, const float* b1,
                                      const float* W2, const float* b2, const int32_t* drop_bits, float drop_p, int64_t B,
                                      int64_t H, int64_t W, int64_t kh, int64_t kw, float* g_x_cl, float* g_W1, float* g_b1,
                                      float* g_W2, float* g_b2, void* workspace, int64_t workspace_bytes, void* stream) {
  // g_W1 = g_b1 = g_W2 = g_b2 = NULL: input gradient only (no workspace needed)
  const bool wgrad = g_W1 || g_b1 || g_W2 || g_b2;
  MLG_CHECK_ARG(g_a0 && x_cl && W1 && b1 && W2 && b2 && g_x_cl && (!wgrad || (g_W1 && g_b1 && g_W2 && g_b2 && workspace)),
                "mlg_head_conv_pool_bwd: null pointer");
  MLG_CHECK_ARG(B >= 1 && H >= 1 && W >= 1 && kh >= 1 && kw >= 1 && kh <= H && kw <= W, "mlg_head_conv_pool_bwd: bad sizes");
  MLG_CHECK_ARG(drop_p == 0.f || drop_bits, "mlg_head_conv_pool_bwd: dropout needs drop_bits");
  ConvPoolP P;
  if (int rc = conv_pool_fill(P, x_cl, W1, b1, W2, b2, drop_bits, drop_p, B, H, W, kh, kw)) return rc;
  MLG_CHECK_ARG(!wgrad || workspace_bytes >= mlg_head_conv_pool_bwd_workspace_bytes(B, H, W, kh, kw),
                "mlg_head_conv_pool_bwd: workspace too small");
  MLG_CHECK_ARG((uintptr_t)g_x_cl % 16 == 0, "mlg_head_conv_pool_bwd: g_x_cl must be 16-byte aligned");
  P.ld = ld; P.g_a0 = g_a0; P.g_x = g_x_cl; P.partial = wgrad ? (float*)workspace : nullptr;
  const int blocks = conv_pool_blocks(P);
  const size_t smem = conv_pool_smem(P, true);
  MLG_CHECK_ARG(smem <= 227 * 1024, "mlg_head_conv_pool_bwd: %lld windows per block do not fit shared memory", (long long)P.NB * P.Wo);
  cudaStream_t st = (cudaStream_t)stream;
  MLG_CUDA(cudaFuncSetAttribute(head_conv_pool_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  head_conv_pool_bwd_kernel<<<blocks, kPix, smem, st>>>(P);
  MLG_CHECK_LAUNCH("mlg_head_conv_pool_bwd");
  if (P.Ho * P.kh < P.H) {
    const long long n4 = (long long)B * (P.H - P.Ho * P.kh) * P.W * (CIN / 4);
    head_conv_tail_zero_kernel<<<(unsigned)((n4 + 255) / 256 > 1024 ? 1024 : (n4 + 255) / 256), 256, 0, st>>>(
        reinterpret_cast<float4*>(g_x_cl), (int)B, P.H, P.W, P.Ho * P.kh);
    MLG_CHECK_LAUNCH("mlg_head_conv_pool_bwd(tail)");
  }
  if (wgrad) {
    head_conv_reduce_kernel<<<mlg_ceil_div(kGradFloats, 128), 128, 0, st>>>(P.partial, blocks, g_W1, g_b1, g_W2, g_b2);
    MLG_CHECK_LAUNCH("mlg_head_conv_pool_bwd(reduce)");
  }
  return MLG_OK;
}

extern "C" int64_t mlg_head_mlp_workspace_bytes(int64_t R, int64_t D, int64_t K) {
  return ((int64_t)mlp_fwd_slices(K) * R * D + R + 4) * 4;
}

extern "C" int mlg_head_mlp_fwd(const float* a0, int64_t ld_a, const float* W0, const float* b0, const float* W3,
                                const float* b3, const int32_t* drop_bits, float drop_p, const float* y, const float* weight,
                                int64_t R, int64_t D, int64_t K, float* a1, float* pred, float* loss, void* workspace,
                                int64_t workspace_bytes, void* stream) {
  MLG_CHECK_ARG(a0 && W0 && b0 && W3 && b3 && a1 && pred && workspace, "mlg_head_mlp_fwd: null pointer");
  MLG_CHECK_ARG(R >= 1 && R <= 64 && D >= 32 && D % 32 == 0 && D <= 512 && K >= 1 && ld_a >= K,
                "mlg_head_mlp_fwd: need 1 <= rows <= 64 (got %lld), D a multiple of 32 up to 512 (got %lld)", (long long)R, (long long)D);
  MLG_CHECK_ARG(!y || loss, "mlg_head_mlp_fwd: y given without a loss output");
  MLG_CHECK_ARG(drop_p >= 0.f && drop_p < 1.f && (drop_p == 0.f || drop_bits), "mlg_head_mlp_fwd: bad dropout arguments");
  MLG_CHECK_ARG(workspace_bytes >= mlg_head_mlp_workspace_bytes(R, D, K), "mlg_head_mlp_fwd: workspace too small");
  MlpP P;
  memset(&P, 0, sizeof(P));
  P.a0 = a0; P.W0 = W0; P.b0 = b0; P.W3 = W3; P.b3 = b3;
  P.bits = drop_p > 0.f ? drop_bits : nullptr;
  P.thr = drop_threshold(drop_p); P.keep_scale = 1.f / (1.f - drop_p);
  P.y = y; P.weight = weight;
  P.R = (int)R; P.D = (int)D; P.K = (int)K; P.ld_a = ld_a;
  P.slices = mlp_fwd_slices(K);
  P.partial = (float*)workspace;
  P.rowloss = P.partial + (size_t)P.slices * R * D;
  P.counter = (unsigned*)(P.rowloss + R);
  P.a1 = a1; P.pred = pred; P.loss = loss;
  cudaStream_t st = (cudaStream_t)stream;
  const int RT = R <= 32 ? 32 : 64;
  const size_t smem = ((size_t)NG * WG_LD + (size_t)KG * RT) * 4;
  dim3 grid((unsigned)((D + NG - 1) / NG), (unsigned)P.slices);
  if (RT == 32) {
    MLG_CUDA(cudaFuncSetAttribute(head_mlp_partial_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    head_mlp_partial_kernel<32><<<grid, 256, smem, st>>>(P);
  } else {
    MLG_CUDA(cudaFuncSetAttribute(head_mlp_partial_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    head_mlp_partial_kernel<64><<<grid, 256, smem, st>>>(P);
  }
  MLG_CHECK_LAUNCH("mlg_head_mlp_fwd(partial)");
  head_mlp_finish_kernel<<<(unsigned)R, kThreads, 0, st>>>(P);
  MLG_CHECK_LAUNCH("mlg_head_mlp_fwd(finish)");
  return MLG_OK;
}

extern "C" int mlg_head_mlp_bwd(const float* g_pred, const float* g_loss, const float* pred, const float* y,
                                const float* weight, const float* a0, int64_t ld_a, const float* a1, const float* W0,
                                const float* W3, float drop_p, int64_t R, int64_t D, int64_t K, float* g_a0, int64_t ld_g,
                                float* g_W0, float* g_b0, float* g_W3, float* g_b3, void* stream) {
  // g_W0 = g_b0 = g_W3 = g_b3 = NULL: input gradient only (one pass over W0 instead of two)
  const bool wgrad = g_W0 || g_b0 || g_W3 || g_b3;
  MLG_CHECK_ARG(pred && a0 && a1 && W0 && W3 && (!wgrad || (g_W0 && g_b0 && g_W3 && g_b3)), "mlg_head_mlp_bwd: null pointer");
  MLG_CHECK_ARG(wgrad || g_a0, "mlg_head_mlp_bwd: no output requested");
  MLG_CHECK_ARG(g_pred || g_loss, "mlg_head_mlp_bwd: neither g_pred nor g_loss given");
  MLG_CHECK_ARG(!g_loss || y, "mlg_head_mlp_bwd: g_loss needs y");
  MLG_CHECK_ARG(R >= 1 && R <= 64 && D >= 32 && D % 32 == 0 && D <= 512 && K >= 1, "mlg_head_mlp_bwd: need rows <= 64, D a multiple of 32 up to 512");
  MLG_CHECK_ARG(ld_a >= K && (!g_a0 || ld_g >= K), "mlg_head_mlp_bwd: leading dimension too small");
  MlpBwdP P;
  memset(&P, 0, sizeof(P));
  P.g_pred = g_pred; P.g_loss = g_loss; P.pred = pred; P.y = y; P.weight = weight;
  P.a0 = a0; P.a1 = a1; P.W0 = W0; P.W3 = W3;
  P.R = (int)R; P.D = (int)D; P.K = (int)K; P.ld_a = ld_a; P.ld_g = ld_g;
  P.keep_scale = 1.f / (1.f - drop_p);
  P.g_a0 = g_a0; P.g_W0 = g_W0; P.g_b0 = g_b0; P.g_W3 = g_W3; P.g_b3 = g_b3;
  const int RT = R <= 32 ? 32 : 64, ks = mlp_ks(R, D);
  const size_t smem = ((size_t)D * (ks + 1) + (size_t)ks * RT + (size_t)RT * D + 2 * RT) * 4;
  MLG_CHECK_ARG(smem <= 227 * 1024, "mlg_head_mlp_bwd: %lld rows x %lld hidden units exceed shared memory", (long long)R, (long long)D);
  const int threads = D < 256 ? 256 : (int)D;
  const int ngrp = threads / ks;
  MLG_CHECK_ARG(mlp_bwd_rows_per_group(RT, ngrp) * ngrp >= RT, "mlg_head_mlp_bwd: %d row groups of at most 16 rows do not cover %d rows",
                ngrp, RT);
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned blocks = (unsigned)mlp_slices(R, D, K);
#define MLG_MLP_B(RR, KK)                                                                                                \
  do {                                                                                                                   \
    MLG_CUDA(cudaFuncSetAttribute(head_mlp_bwd_kernel<RR, KK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    head_mlp_bwd_kernel<RR, KK><<<blocks, (unsigned)threads, smem, st>>>(P);                                            \
  } while (0)
  if (RT == 32) MLG_MLP_B(32, 64);
  else if (ks == 64) MLG_MLP_B(64, 64);
  else MLG_MLP_B(64, 32);
#undef MLG_MLP_B
  MLG_CHECK_LAUNCH("mlg_head_mlp_bwd");
  return MLG_OK;
}
