// Expected gradients (Erion et al., Nature Machine Intelligence 2021) against a background cohort (sm_100a):
//     phi_i(x) = E_{x' ~ bank, alpha ~ U(0,1)} [ (x_i - x'_i) * dF/dx_i (x' + alpha (x - x')) ]
// Each slot s of a replay holds one draw (j_s, alpha_s) of a patient; the host draws them (attribution.eg_draws).
//
// mlg_attr_eg_interp: out[s,:] = fmaf(alpha_s, x[s,:], (1 - alpha_s) * bank[j_s,:]), the interpolant the captured forward
//     reads.  alpha = 1 gives x and alpha = 0 the bank row, bitwise (0 * v and 1 * v are exact; v + 0 = v).
// mlg_attr_eg_accumulate: acc[p,:] (+)= sum_{s in slots of p} w_s * (x[s,:] - bank[j_s,:]) * g[s,:], slots in order: the
//     Monte-Carlo sum without a [slots, N] difference tensor.  One thread per output element, no atomics, so a patient's
//     result has the same bits wherever its slots sit.
// A j outside [0, M) is not read: its row becomes NaN and *bad is set to 1, for the host to check at its next synchronisation.
#include <cmath>

#include "common.cuh"
#include "../../include/mlg_b200.h"

namespace {

__global__ void eg_interp_kernel(const float* __restrict__ x, const float* __restrict__ bank, long long M,
                                 const int* __restrict__ j, const float* __restrict__ alpha, long long N,
                                 float* __restrict__ out, int* __restrict__ bad) {
  const long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x;   // grid: (columns, slots)
  const int s = blockIdx.y;
  if (c >= N) return;
  const size_t i = (size_t)s * N + c;
  const int js = __ldg(j + s);
  if (js < 0 || js >= M) {
    out[i] = NAN;
    *bad = 1;
    return;
  }
  const float a = __ldg(alpha + s);
  out[i] = fmaf(a, __ldg(x + i), (1.f - a) * __ldg(bank + (size_t)js * N + c));
}

__global__ void eg_accumulate_kernel(const float* __restrict__ g, const float* __restrict__ x, const float* __restrict__ bank,
                                     long long M, const int* __restrict__ j, const float* __restrict__ w,
                                     const int* __restrict__ slot_ptr, long long N, int accumulate,
                                     float* __restrict__ acc, int* __restrict__ bad) {
  const long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x;   // grid: (columns, outputs)
  const int p = blockIdx.y;
  if (c >= N) return;
  const size_t i = (size_t)p * N + c;
  float s = accumulate ? acc[i] : 0.f;
  const int beg = __ldg(slot_ptr + p), end = __ldg(slot_ptr + p + 1);
  for (int k = beg; k < end; ++k) {
    const int jk = __ldg(j + k);
    if (jk < 0 || jk >= M) {
      s = NAN;
      *bad = 1;
      continue;
    }
    const float d = __ldg(x + (size_t)k * N + c) - __ldg(bank + (size_t)jk * N + c);
    s = fmaf(__ldg(w + k) * d, __ldg(g + (size_t)k * N + c), s);
  }
  acc[i] = s;
}

}  // namespace

extern "C" int mlg_attr_eg_interp(const float* x, const float* bank, int64_t M, const int32_t* j, const float* alpha, int64_t B,
                                  int64_t N, float* out, int32_t* bad, void* stream) {
  MLG_CHECK_ARG(x && bank && j && alpha && out && bad, "mlg_attr_eg_interp: null pointer");
  MLG_CHECK_ARG(M >= 1 && B >= 1 && B <= 65535 && N >= 1 && B * N < (1ll << 40) && M * N < (1ll << 40),
                "mlg_attr_eg_interp: bad sizes");
  const dim3 grid(mlg_ceil_div(N, 256), (unsigned)B);
  eg_interp_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, bank, M, j, alpha, N, out, bad);
  MLG_CHECK_LAUNCH("mlg_attr_eg_interp");
  return MLG_OK;
}

extern "C" int mlg_attr_eg_accumulate(const float* g, const float* x, const float* bank, int64_t M, const int32_t* j,
                                      const float* w, const int32_t* slot_ptr, int64_t n_out, int64_t N, int accumulate,
                                      float* acc, int32_t* bad, void* stream) {
  MLG_CHECK_ARG(g && x && bank && j && w && slot_ptr && acc && bad, "mlg_attr_eg_accumulate: null pointer");
  MLG_CHECK_ARG(M >= 1 && n_out >= 1 && n_out <= 65535 && N >= 1 && n_out * N < (1ll << 40) && M * N < (1ll << 40),
                "mlg_attr_eg_accumulate: bad sizes");
  const dim3 grid(mlg_ceil_div(N, 256), (unsigned)n_out);
  eg_accumulate_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(g, x, bank, M, j, w, slot_ptr, N, accumulate, acc, bad);
  MLG_CHECK_LAUNCH("mlg_attr_eg_accumulate");
  return MLG_OK;
}
