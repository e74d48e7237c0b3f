// Shared helpers for libpcb200 (sm_100a).  Not part of the public ABI.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include "../../include/pcb200.h"

namespace pcb {

void set_error(const char* fmt, ...);
extern std::atomic<uint64_t> g_launches;

inline int check_launch(const char* what) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("%s: %s", what, cudaGetErrorString(e)); return PCB_ERR_CUDA; }
  return PCB_OK;
}
#define PCB_CUDA(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { pcb::set_error("%s: %s", #call, cudaGetErrorString(e_)); return PCB_ERR_CUDA; } } while (0)
#define PCB_ARG(cond) do { if (!(cond)) { pcb::set_error("bad argument: %s (%s:%d)", #cond, __FILE__, __LINE__); return PCB_ERR_ARG; } } while (0)

constexpr uint64_t KEY_EMPTY = 0xFFFFFFFFFFFFFFFFull;
constexpr int COORD_BIAS = 32768;

__host__ __device__ __forceinline__ uint64_t mix64(uint64_t k) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdULL; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ULL; k ^= k >> 33; return k;
}

__device__ __forceinline__ int hash_lookup(const uint64_t* __restrict__ tk, const int32_t* __restrict__ tv,
                                           uint64_t mask, uint64_t key) {
  uint64_t slot = mix64(key) & mask;
  while (true) {
    uint64_t k = tk[slot];
    if (k == key) return tv[slot];
    if (k == KEY_EMPTY) return -1;
    slot = (slot + 1) & mask;
  }
}

// Optional per-launch timing (pcb_profile_*, unit.cu): CUDA events around every convolution / weight-gradient entry point.
void prof_begin(cudaStream_t st);
// kind: 0 conv forward / data gradient, 1 weight gradient, 2 BatchNorm forward pass(es) of a unit, 3 BatchNorm backward of a unit,
// 4 PointInfoNCE forward + backward, 5 SGD step, 6 weight re-tiling
void prof_end(cudaStream_t st, int kind);
struct ProfScope {
  cudaStream_t st; int kind;
  ProfScope(cudaStream_t s, int k) : st(s), kind(k) { prof_begin(st); }
  ~ProfScope() { prof_end(st, kind); }
};

// Programmatic dependent launch (default; PCB_PDL=0 turns it off): every kernel below starts with pdl_wait() -- it blocks until the preceding kernel of
// the stream has completed and its writes are visible -- followed by pdl_trigger(), which lets the NEXT kernel's CTAs be scheduled
// as soon as all of this kernel's CTAs are running.  The launch latency and CTA ramp-up of a kernel then overlap the tail of its
// predecessor; ordering is unchanged (nothing precedes the wait).  Launched without the attribute, both are no-ops.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
bool pdl_enabled();

template <typename... Exp, typename... Act>
inline void launch_kernel(void (*kernel)(Exp...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Act&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl_enabled() ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kernel, static_cast<Act&&>(args)...);       // errors surface through check_launch (cudaGetLastError)
}

// Logsumexp of a row of C fp32 values shared by W lanes of a warp (lane strides by W; W = 32: one warp per row, W = 1: one thread per
// row): m = max, s = sum of exp(x - m), returns m + log(s).  The cross-entropy (loss.cu) and segmentation-metric (seg_eval.cu) rows.
template <int W>
__device__ __forceinline__ float row_logsumexp(const float* __restrict__ x, int C, int lane, float& m, float& s) {
  m = -INFINITY;
  for (int c = lane; c < C; c += W) m = fmaxf(m, x[c]);
  for (int o = W / 2; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  s = 0.f;
  for (int c = lane; c < C; c += W) s += expf(x[c] - m);
  for (int o = W / 2; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  return m + logf(s);
}

inline int current_device() { int dev = 0; cudaGetDevice(&dev); return (dev >= 0 && dev < 64) ? dev : 0; }

inline int num_sms() {
  static int n[64] = {};
  const int dev = current_device();
  if (!n[dev]) { cudaDeviceGetAttribute(&n[dev], cudaDevAttrMultiProcessorCount, dev); if (n[dev] <= 0) n[dev] = 148; }
  return n[dev];
}

}  // namespace pcb
