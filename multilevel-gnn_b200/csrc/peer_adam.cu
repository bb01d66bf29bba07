// Data-parallel optimizer step as ONE kernel over NVLink / NVSwitch peer memory (sm_100a):
//     reduce-scatter(gradients) -> Adam on the owned shard -> all-gather(parameters)
// The reference trains on one device (train.py:38-68: loss.backward(); optimizer.step()); patient graphs are independent,
// so the data-parallel wrapper (SURVEY.md section 8e) only has to average the gradients.  Instead of an NCCL all-reduce
// followed by a replicated Adam, every rank keeps its flat gradient bucket, its flat parameter buffer and a small flag
// block in a cudaMalloc'ed arena that is mapped into every other rank of the box (CUDA IPC), and this kernel
//   0. tells every peer "my gradients of step e are final" and waits for the same from all of them,
//   1. for the 1/world shard it owns: loads that slice of every peer's gradients straight over NVLink (fixed rank order
//      0..world-1, so every replica gets bitwise-identical parameters), averages, applies torch.optim.Adam's update to
//      its shard of the optimizer state, and stores the new parameter values into EVERY peer's parameter buffer,
//   2. tells every peer "my writes of step e are done" and waits for the same from all before it retires.
// No gradient is ever written back, Adam state exists once per box (ZeRO-1), and since it is an ordinary kernel launch
// with fixed pointers the whole training step (forward, loss, backward, this kernel) is ONE CUDA graph per rank.
// Per-GPU traffic: (world-1)/world * 4n bytes read and the same written over NVLink + 16 B/parameter of local state.
//
// Flag block (uint32, one per rank, peer-writable):  [0..7] ready[src]   [8..15] done[src]   [16] epoch   [17] block
// counter   [18] status.  A wait that exceeds the timeout is a HARD failure: the rank sets its own status word, the status
// word of EVERY peer and the host-visible status word (pinned memory), skips the update (parameters and optimizer state stay
// untouched, so the replicas do not silently diverge) and every later launch returns immediately; the host (Trainer.step)
// reads the pinned word before each step and raises on all ranks.
#include <cooperative_groups.h>

#include "common.cuh"
#include "../../include/mlg_b200.h"

namespace {

constexpr int kMaxWorld = 8;
constexpr int kThreads = 512;
constexpr int F_READY = 0, F_DONE = 8, F_EPOCH = 16, F_COUNT = 17, F_STATUS = 18;

struct PeerP {
  const float* grad[kMaxWorld];
  float* param[kMaxWorld];
  unsigned* flags[kMaxWorld];
  float* m;          // exp_avg of the owned shard      [hi - lo]
  float* v;          // exp_avg_sq of the owned shard   [hi - lo]
  float* step_dev;   // Adam step counter (float, as mlg_adam_step)
  int* host_status;  // pinned host word (or NULL)
  long long lo, hi;  // owned shard, multiples of 4
  int world, rank;
  float lr, b1, b2, eps, wd;
  long long timeout_clocks;
};

__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float4 ld_peer4(const float* p) {   // never cached: the owner rewrites it every step
  float4 v;
  asm volatile("ld.volatile.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}

// a failed wait: sticky on this rank, broadcast to every peer and to the host
__device__ __forceinline__ void fail_everywhere(const PeerP& P) {
  for (int r = 0; r < P.world; ++r) st_release_sys(P.flags[r] + F_STATUS, 1u);
  if (P.host_status) *reinterpret_cast<volatile int*>(P.host_status) = 1;
  __threadfence_system();
}

// wait until flag[i] has reached `epoch` for every rank i < world (threads 0..world-1 poll one flag each); false = gave up
__device__ __forceinline__ bool wait_all(const PeerP& P, unsigned* mine, int base, unsigned epoch, int* shared_ok) {
  if (threadIdx.x == 0) *shared_ok = 1;
  __syncthreads();
  if ((int)threadIdx.x < P.world) {
    const unsigned* f = mine + base + threadIdx.x;
    const long long t0 = clock64();
    while ((int)(ld_acquire_sys(f) - epoch) < 0) {
      if (clock64() - t0 > P.timeout_clocks || ld_acquire_sys(mine + F_STATUS) != 0u) {
        *shared_ok = 0;
        break;
      }
      __nanosleep(64);
    }
  }
  __syncthreads();
  return *shared_ok != 0;
}

__device__ __forceinline__ void adam_one(float& p, float g, float& m, float& v, float b1, float b2, float eps, float wd,
                                         float step_size, float inv_sqrt_bc2) {
  if (wd != 0.f) g = fmaf(wd, p, g);
  m = fmaf(b1, m, (1.f - b1) * g);
  v = fmaf(b2, v, (1.f - b2) * g * g);
  const float denom = sqrtf(v) * inv_sqrt_bc2 + eps;     // torch: (sqrt(v) / sqrt(bias_correction2)) + eps
  p -= step_size * (m / denom);
}

__device__ __forceinline__ void peer_adam_body(const PeerP& P, int block, int nblocks) {
  __shared__ int is_last, ok;
  unsigned* mine = P.flags[P.rank];
  const int world = P.world;
  if (*reinterpret_cast<volatile unsigned*>(mine + F_STATUS) != 0u) return;   // sticky failure: do nothing
  // the epoch word is only advanced by the LAST block of a run, after every block of that run has read it
  const unsigned epoch = *reinterpret_cast<volatile unsigned*>(mine + F_EPOCH) + 1u;

  // ---- 0. gradients of every rank are final ----
  if (block == 0 && (int)threadIdx.x < world) {
    __threadfence_system();
    st_release_sys(P.flags[threadIdx.x] + F_READY + P.rank, epoch);
  }
  if (!wait_all(P, mine, F_READY, epoch, &ok)) {
    if (threadIdx.x == 0) fail_everywhere(P);
    return;                      // parameters and optimizer state untouched
  }

  // ---- 1. owned shard: sum over ranks in rank order, Adam, broadcast the new values ----
  const float t = *reinterpret_cast<volatile float*>(P.step_dev) + 1.f;
  const float bc1 = 1.f - powf(P.b1, t), bc2 = 1.f - powf(P.b2, t);
  const float step_size = P.lr / bc1, inv_sqrt_bc2 = 1.f / sqrtf(bc2);
  const float inv_world = 1.f / (float)world;
  const long long stride = (long long)nblocks * kThreads * 4;
  for (long long i = P.lo + ((long long)block * kThreads + threadIdx.x) * 4; i < P.hi; i += stride) {
    float4 g[kMaxWorld];
#pragma unroll
    for (int r = 0; r < kMaxWorld; ++r)
      if (r < world) g[r] = ld_peer4(P.grad[r] + i);
    float4 s = g[0];
#pragma unroll
    for (int r = 1; r < kMaxWorld; ++r)
      if (r < world) {
        s.x += g[r].x; s.y += g[r].y; s.z += g[r].z; s.w += g[r].w;
      }
    s.x *= inv_world; s.y *= inv_world; s.z *= inv_world; s.w *= inv_world;
    const long long j = i - P.lo;
    float4 pi = *reinterpret_cast<const float4*>(P.param[P.rank] + i);
    float4 mi = *reinterpret_cast<const float4*>(P.m + j), vi = *reinterpret_cast<const float4*>(P.v + j);
    adam_one(pi.x, s.x, mi.x, vi.x, P.b1, P.b2, P.eps, P.wd, step_size, inv_sqrt_bc2);
    adam_one(pi.y, s.y, mi.y, vi.y, P.b1, P.b2, P.eps, P.wd, step_size, inv_sqrt_bc2);
    adam_one(pi.z, s.z, mi.z, vi.z, P.b1, P.b2, P.eps, P.wd, step_size, inv_sqrt_bc2);
    adam_one(pi.w, s.w, mi.w, vi.w, P.b1, P.b2, P.eps, P.wd, step_size, inv_sqrt_bc2);
    *reinterpret_cast<float4*>(P.m + j) = mi;
    *reinterpret_cast<float4*>(P.v + j) = vi;
#pragma unroll
    for (int r = 0; r < kMaxWorld; ++r)
      if (r < world) *reinterpret_cast<float4*>(P.param[r] + i) = pi;
  }

  // ---- 2. every rank's parameter writes have landed ----
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned c = atomicAdd(mine + F_COUNT, 1u);
    __threadfence();
    is_last = (c == (unsigned)nblocks - 1);
  }
  __syncthreads();
  if (!is_last) return;
  if ((int)threadIdx.x < world) {
    __threadfence_system();
    st_release_sys(P.flags[threadIdx.x] + F_DONE + P.rank, epoch);
  }
  const bool done = wait_all(P, mine, F_DONE, epoch, &ok);
  if (threadIdx.x == 0) {
    if (!done) fail_everywhere(P);
    mine[F_COUNT] = 0u;
    *reinterpret_cast<volatile float*>(P.step_dev) = t;
    __threadfence();
    *reinterpret_cast<volatile unsigned*>(mine + F_EPOCH) = epoch;
  }
}

__global__ void __launch_bounds__(kThreads) peer_adam_kernel(const PeerP P) { peer_adam_body(P, blockIdx.x, gridDim.x); }

// TEST SUPPORT: all ranks of a job as ONE cooperative launch on one GPU (blockIdx.y = rank), so that the blocks that wait on
// one another are guaranteed co-resident (separate launches on one GPU are not: B200_PROFILING.md)
__global__ void __launch_bounds__(kThreads) peer_adam_emulated_kernel(const PeerP* __restrict__ ranks) {
  __shared__ PeerP P;
  if (threadIdx.x == 0) P = ranks[blockIdx.y];
  __syncthreads();
  peer_adam_body(P, blockIdx.x, gridDim.x);
}

int fill_peer(PeerP& P, const float* const* peer_grads, float* const* peer_params, void* const* peer_flags, int world, int rank,
              int64_t n, float* exp_avg, float* exp_avg_sq, float* step_dev, float lr, float beta1, float beta2,
              float eps, float weight_decay, double timeout_s, int* host_status) {
  MLG_CHECK_ARG(peer_grads && peer_params && peer_flags && exp_avg && exp_avg_sq && step_dev, "mlg_peer_adam_step: null pointer");
  MLG_CHECK_ARG(world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world, "mlg_peer_adam_step: world must be 1..8");
  MLG_CHECK_ARG(n >= 0 && n % (4 * world) == 0, "mlg_peer_adam_step: the bucket must hold a multiple of 4*world elements");
  memset(&P, 0, sizeof(P));
  for (int r = 0; r < world; ++r) {
    MLG_CHECK_ARG(peer_grads[r] && peer_params[r] && peer_flags[r], "mlg_peer_adam_step: null peer pointer");
    MLG_CHECK_ARG(((uintptr_t)peer_grads[r] | (uintptr_t)peer_params[r]) % 16 == 0, "mlg_peer_adam_step: 16-byte alignment");
    P.grad[r] = peer_grads[r];
    P.param[r] = peer_params[r];
    P.flags[r] = (unsigned*)peer_flags[r];
  }
  MLG_CHECK_ARG(((uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) % 16 == 0, "mlg_peer_adam_step: 16-byte alignment");
  const long long shard = n / world;
  P.m = exp_avg; P.v = exp_avg_sq; P.step_dev = step_dev; P.host_status = host_status;
  P.lo = shard * rank; P.hi = P.lo + shard;
  P.world = world; P.rank = rank;
  P.lr = lr; P.b1 = beta1; P.b2 = beta2; P.eps = eps; P.wd = weight_decay;
  P.timeout_clocks = (long long)((timeout_s > 0 ? timeout_s : 5.0) * 1.9e9);
  return MLG_OK;
}

}  // namespace

extern "C" int64_t mlg_peer_flag_bytes(void) { return 256; }

extern "C" void* mlg_peer_alloc(int64_t bytes) {
  void* p = nullptr;
  if (bytes <= 0) return nullptr;
  cudaError_t e = cudaMalloc(&p, (size_t)bytes);
  if (e != cudaSuccess) {
    mlg_set_error("mlg_peer_alloc(%lld): %s", (long long)bytes, cudaGetErrorString(e));
    return nullptr;
  }
  e = cudaMemset(p, 0, (size_t)bytes);
  if (e != cudaSuccess) {
    mlg_set_error("mlg_peer_alloc: memset: %s", cudaGetErrorString(e));
    cudaFree(p);
    return nullptr;
  }
  return p;
}

extern "C" int mlg_peer_free(void* ptr) {
  if (ptr && cudaFree(ptr) != cudaSuccess) {
    mlg_set_error("mlg_peer_free: %s", cudaGetErrorString(cudaGetLastError()));
    return MLG_ERR_CUDA;
  }
  return MLG_OK;
}

extern "C" int mlg_peer_export(void* ptr, void* handle64) {
  MLG_CHECK_ARG(ptr && handle64, "mlg_peer_export: null pointer");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  cudaError_t e = cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(handle64), ptr);
  if (e != cudaSuccess) {
    mlg_set_error("mlg_peer_export: %s", cudaGetErrorString(e));
    return MLG_ERR_CUDA;
  }
  return MLG_OK;
}

extern "C" void* mlg_peer_open(const void* handle64) {
  if (!handle64) return nullptr;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, sizeof(h));
  void* p = nullptr;
  cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) {
    mlg_set_error("mlg_peer_open: %s", cudaGetErrorString(e));
    cudaGetLastError();
    return nullptr;
  }
  return p;
}

extern "C" int mlg_peer_close(void* ptr) {
  if (ptr && cudaIpcCloseMemHandle(ptr) != cudaSuccess) {
    mlg_set_error("mlg_peer_close: %s", cudaGetErrorString(cudaGetLastError()));
    return MLG_ERR_CUDA;
  }
  return MLG_OK;
}

extern "C" int mlg_peer_adam_step(const float* const* peer_grads, float* const* peer_params, void* const* peer_flags,
                                  int world, int rank, int64_t n, float* exp_avg, float* exp_avg_sq,
                                  float* step_dev, float lr, float beta1, float beta2, float eps, float weight_decay,
                                  double timeout_s, int32_t* host_status, void* stream) {
  if (n == 0) return MLG_OK;
  PeerP P;
  if (int rc = fill_peer(P, peer_grads, peer_params, peer_flags, world, rank, n, exp_avg, exp_avg_sq, step_dev, lr, beta1,
                         beta2, eps, weight_decay, timeout_s, host_status))
    return rc;
  // enough blocks to keep ~world float4 loads per thread in flight on every NVLink, few enough that the whole grid is
  // resident next to whatever else the stream overlaps
  long long blocks = ((P.hi - P.lo) / 4 + kThreads - 1) / kThreads;
  if (blocks > 96) blocks = 96;
  if (blocks < 1) blocks = 1;
  peer_adam_kernel<<<(unsigned)blocks, kThreads, 0, (cudaStream_t)stream>>>(P);
  MLG_CHECK_LAUNCH("mlg_peer_adam_step");
  return MLG_OK;
}

// TEST SUPPORT (single GPU): `world` ranks whose arenas live on this device, stepped by ONE cooperative launch.
// peer_* tables: world pointers each, shared by all ranks; exp_avg / exp_avg_sq / step_dev: one per rank.
// ranks_dev: device scratch of mlg_peer_emulated_bytes(world) bytes.
extern "C" int64_t mlg_peer_emulated_bytes(int world) { return (int64_t)world * (int64_t)sizeof(PeerP); }

extern "C" int mlg_peer_adam_step_emulated(const float* const* peer_grads, float* const* peer_params, void* const* peer_flags,
                                           int world, int64_t n, float* const* exp_avg, float* const* exp_avg_sq,
                                           float* const* step_dev, float lr, float beta1, float beta2, float eps,
                                           float weight_decay, double timeout_s, void* ranks_dev, void* stream) {
  MLG_CHECK_ARG(exp_avg && exp_avg_sq && step_dev && ranks_dev, "mlg_peer_adam_step_emulated: null pointer");
  if (n == 0) return MLG_OK;
  PeerP host[kMaxWorld];
  for (int r = 0; r < world; ++r)
    if (int rc = fill_peer(host[r], peer_grads, peer_params, peer_flags, world, r, n, exp_avg[r], exp_avg_sq[r], step_dev[r],
                           lr, beta1, beta2, eps, weight_decay, timeout_s, nullptr))
      return rc;
  cudaStream_t st = (cudaStream_t)stream;
  MLG_CUDA(cudaMemcpyAsync(ranks_dev, host, sizeof(PeerP) * world, cudaMemcpyHostToDevice, st));
  MLG_CUDA(cudaStreamSynchronize(st));            // `host` is a stack array
  int per_sm = 0, dev = 0, sms = 0;
  MLG_CUDA(cudaGetDevice(&dev));
  MLG_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  MLG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, peer_adam_emulated_kernel, kThreads, 0));
  long long blocks = ((host[0].hi - host[0].lo) / 4 + kThreads - 1) / kThreads;
  const long long cap = (long long)per_sm * sms / world;
  if (blocks > cap) blocks = cap;
  if (blocks > 32) blocks = 32;
  MLG_CHECK_ARG(blocks >= 1, "mlg_peer_adam_step_emulated: %d ranks do not fit one cooperative launch", world);
  dim3 grid((unsigned)blocks, (unsigned)world);
  const PeerP* arg = (const PeerP*)ranks_dev;
  void* args[] = {(void*)&arg};
  MLG_CUDA(cudaLaunchCooperativeKernel((void*)peer_adam_emulated_kernel, grid, dim3(kThreads), args, 0, st));
  return MLG_OK;
}

extern "C" int mlg_peer_status(const void* flags, int* status_out) {
  MLG_CHECK_ARG(flags && status_out, "mlg_peer_status: null pointer");
  unsigned s = 0;
  cudaError_t e = cudaMemcpy(&s, (const unsigned*)flags + F_STATUS, sizeof(s), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) {
    mlg_set_error("mlg_peer_status: %s", cudaGetErrorString(e));
    return MLG_ERR_CUDA;
  }
  *status_out = (int)s;
  return MLG_OK;
}
