// Semantic-segmentation metrics of one batch (`downstream/semseg/lib/test.py:119-149`, `lib/utils.py:117-133`): prediction, cross-entropy,
// precision@1, confusion histogram and per-class average precision, all on the device.
//
//   seg_rows_kernel   tiles of 256 rows staged through shared memory (coalesced); one thread per row: max / first argmax / logsumexp,
//                     the CE term, the correct flag, the histogram bin (privatised per CTA, flushed with integer atomics), the softmax
//                     and one 64-bit sort key per (row, class):  class << 33 | ~bits(prob) << 1 | is_positive.
//   cub radix sort    on bits [0, 33 + ceil(log2 C)): every class becomes one run of n keys, probabilities descending, equal
//                     probabilities (a tie group) adjacent.  prob >= +0, so the fp32 bit order is the value order.
//   ap_flags_kernel   per sorted position: (positive bit, its index if it starts a tie group else 0)
//   cub scan          (sum, max) of those pairs: the true positives up to each position and the start of its tie group.
//   ap_terms_kernel   at each tie-group end e (start s):  (TP_e - TP_{s-1}) * TP_e / (e + 1), fp64, per-CTA partial per class.
//   seg_final_kernel  fixed-order sums of the partials: stats[4] and ap[c] = sum / P_c (NaN when class c has no positive).
// Every floating-point reduction has a fixed order and the histogram uses integer atomics, so two calls are bit-identical.
#include <cub/cub.cuh>
#include "common.cuh"

using namespace pcb;

namespace {

constexpr int ROWS = 256;            // rows per tile == threads of the row pass
constexpr int ROW_CTAS_MAX = 592;    // the row pass is persistent over tiles; fixed cap keeps the partial count device-independent
constexpr int AP_THREADS = 256, AP_ITEMS = 8, AP_CHUNK = AP_THREADS * AP_ITEMS;

inline size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }
__host__ __device__ inline int row_ld(int C) { return C | 1; }           // odd row stride: thread-per-row reads of the tile hit distinct banks
inline int row_ctas(int64_t n) { int64_t t = (n + ROWS - 1) / ROWS; return (int)(t < ROW_CTAS_MAX ? t : ROW_CTAS_MAX); }
inline int ap_chunks(int64_t n) { return (int)((n + AP_CHUNK - 1) / AP_CHUNK); }
inline int key_bits(int C) { int b = 0; while ((1 << b) < C) ++b; return 33 + b; }
inline size_t rows_smem(int C) { return (size_t)ROWS * row_ld(C) * sizeof(float) + (size_t)C * C * sizeof(int); }

__device__ __forceinline__ bool valid_target(int64_t t, int C, int64_t ignore) { return t >= 0 && t < C && t != ignore; }

// block-wide sum in a fixed order (warp xor tree, then warps in index order); the result is valid in thread 0
template <typename T>
__device__ T block_sum(T v, T* red) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  T tot = 0;
  if (threadIdx.x == 0)
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += red[w];
  return tot;
}

__global__ void __launch_bounds__(ROWS) seg_rows_kernel(const float* __restrict__ X, const int64_t* __restrict__ target, int64_t n, int C,
                                                         int64_t ignore, int32_t* __restrict__ pred, float* __restrict__ prob,
                                                         uint64_t* __restrict__ keys, unsigned long long* __restrict__ hist,
                                                         double* __restrict__ part_loss, long long* __restrict__ part_cnt) {
  extern __shared__ float sm[];
  const int ld = row_ld(C);
  float* tile = sm;                                        // [ROWS][ld]
  int* hs = reinterpret_cast<int*>(sm + ROWS * ld);        // [C][C]
  __shared__ double red_d[ROWS / 32];
  __shared__ long long red_l[ROWS / 32];
  pdl_wait(); pdl_trigger();
  const int tid = threadIdx.x;
  for (int i = tid; i < C * C; i += ROWS) hs[i] = 0;
  double loss = 0.0;
  long long n_valid = 0, n_correct = 0;
  const int64_t tiles = (n + ROWS - 1) / ROWS;
  for (int64_t tl = blockIdx.x; tl < tiles; tl += gridDim.x) {
    const int64_t r0 = tl * ROWS;
    const int rows = (int)(n - r0 < ROWS ? n - r0 : ROWS);
    const float* src = X + r0 * C;
    __syncthreads();                                       // previous tile's prob store / the histogram zeroing are done
    for (int e = tid; e < rows * C; e += ROWS) { const int r = e / C; tile[r * ld + (e - r * C)] = src[e]; }
    __syncthreads();
    if (tid < rows) {
      const int64_t row = r0 + tid;
      float* x = tile + tid * ld;
      float m, s;
      const float lse = row_logsumexp<1>(x, C, 0, m, s);
      int p = 0;                                           // first maximal index (torch's max(1)[1])
      for (int c = 1; c < C; ++c) p = x[c] > x[p] ? c : p;
      const int64_t t = target[row];
      const bool v = valid_target(t, C, ignore);
      if (v) {
        loss += (double)(lse - x[t]);
        ++n_valid;
        n_correct += (p == (int)t);
        atomicAdd(&hs[(int)t * C + p], 1);
      }
      if (pred) pred[row] = p;
      for (int c = 0; c < C; ++c) {
        const float pc = expf(x[c] - m) / s;
        const uint64_t key = ((uint64_t)c << 33) | ((uint64_t)(~__float_as_uint(pc)) << 1) | (uint64_t)(v && t == c);
        keys[(int64_t)c * n + row] = key;
        x[c] = pc;
      }
    }
    if (prob) {
      __syncthreads();
      float* dst = prob + r0 * C;
      for (int e = tid; e < rows * C; e += ROWS) { const int r = e / C; dst[e] = tile[r * ld + (e - r * C)]; }
    }
  }
  __syncthreads();
  for (int i = tid; i < C * C; i += ROWS)
    if (hs[i]) atomicAdd(hist + i, (unsigned long long)hs[i]);
  const double ls = block_sum(loss, red_d);
  if (tid == 0) part_loss[blockIdx.x] = ls;
  const long long nv = block_sum(n_valid, red_l);
  if (tid == 0) part_cnt[2 * blockIdx.x] = nv;
  const long long nc = block_sum(n_correct, red_l);
  if (tid == 0) part_cnt[2 * blockIdx.x + 1] = nc;
}

__device__ __forceinline__ uint32_t prob_bits(uint64_t key) { return (uint32_t)(key >> 1); }

// f[i] = (positive bit, i if i starts a tie group of its class else 0)
__global__ void ap_flags_kernel(const uint64_t* __restrict__ sk, int64_t n, int64_t total, int2* __restrict__ f) {
  pdl_wait(); pdl_trigger();
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const uint64_t k = sk[i];
  const bool start = (i % n == 0) || prob_bits(sk[i - 1]) != prob_bits(k);
  f[i] = make_int2((int)(k & 1), start ? (int)i : 0);
}

struct SumMax {
  __device__ __forceinline__ int2 operator()(const int2& a, const int2& b) const { return make_int2(a.x + b.x, max(a.y, b.y)); }
};

// grid (chunks, C): CTA (k, c) sums the AP terms of the tie groups of class c that end inside chunk k of its run
__global__ void __launch_bounds__(AP_THREADS) ap_terms_kernel(const uint64_t* __restrict__ sk, const int2* __restrict__ scan, int64_t n,
                                                               double* __restrict__ part_ap) {
  __shared__ double red[AP_THREADS / 32];
  pdl_wait(); pdl_trigger();
  const int c = blockIdx.y;
  const int64_t seg0 = (int64_t)c * n;
  const int base = seg0 > 0 ? scan[seg0 - 1].x : 0;
  double acc = 0.0;
#pragma unroll 2
  for (int j = 0; j < AP_ITEMS; ++j) {
    const int64_t r = (int64_t)blockIdx.x * AP_CHUNK + j * AP_THREADS + threadIdx.x;       // rank within the class run
    if (r >= n) break;
    const int64_t e = seg0 + r;
    if (r + 1 < n && prob_bits(sk[e + 1]) == prob_bits(sk[e])) continue;                 // not the end of its tie group
    const int2 se = scan[e];
    const int tp = se.x - base;
    const int tp_prev = se.y > seg0 ? scan[se.y - 1].x - base : 0;
    if (tp > tp_prev) acc += (double)(tp - tp_prev) * (double)tp / (double)(r + 1);
  }
  const double tot = block_sum(acc, red);
  if (threadIdx.x == 0) part_ap[(int64_t)c * gridDim.x + blockIdx.x] = tot;
}

// stats = {sum CE over valid rows, #valid, #correct, n};  ap[c] = sum of class c's terms / P_c
__global__ void __launch_bounds__(256) seg_final_kernel(const double* __restrict__ part_loss, const long long* __restrict__ part_cnt, int g_rows,
                                                        const double* __restrict__ part_ap, int chunks, const int2* __restrict__ scan, int64_t n,
                                                        int C, double* __restrict__ stats, double* __restrict__ ap) {
  __shared__ double red_d[8];
  __shared__ long long red_l[8];
  pdl_wait(); pdl_trigger();
  double ls = 0.0;
  long long nv = 0, nc = 0;
  for (int i = threadIdx.x; i < g_rows; i += blockDim.x) { ls += part_loss[i]; nv += part_cnt[2 * i]; nc += part_cnt[2 * i + 1]; }
  ls = block_sum(ls, red_d);
  nv = block_sum(nv, red_l);
  nc = block_sum(nc, red_l);
  if (threadIdx.x == 0) { stats[0] = ls; stats[1] = (double)nv; stats[2] = (double)nc; stats[3] = (double)n; }
  const int lane = threadIdx.x & 31;
  for (int c = threadIdx.x >> 5; c < C; c += blockDim.x >> 5) {
    double s = 0.0;
    for (int k = lane; k < chunks; k += 32) s += part_ap[(int64_t)c * chunks + k];
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) {
      const int64_t e = (int64_t)(c + 1) * n - 1;
      const int P = scan[e].x - (c > 0 ? scan[(int64_t)c * n - 1].x : 0);
      ap[c] = P > 0 ? s / (double)P : __longlong_as_double(0x7ff8000000000000ll);
    }
  }
}

size_t cub_bytes(int64_t n, int C) {
  const int total = (int)(n * C);
  size_t a = 0, b = 0;
  cub::DeviceRadixSort::SortKeys(nullptr, a, (const uint64_t*)nullptr, (uint64_t*)nullptr, total, 0, key_bits(C));
  cub::DeviceScan::InclusiveScan(nullptr, b, (const int2*)nullptr, (int2*)nullptr, SumMax(), total);
  return a > b ? a : b;
}

struct Ws { uint64_t* keys; uint64_t* sorted; int2* flags; int2* scan; double* part_loss; long long* part_cnt; double* part_ap; void* cub; size_t cub_bytes; };

Ws carve(void* ws, int64_t n, int C) {
  const size_t nc = (size_t)n * C;
  char* p = (char*)ws;
  Ws w;
  w.keys = (uint64_t*)p; p += align_up(nc * 8);
  w.sorted = (uint64_t*)p; p += align_up(nc * 8);
  w.flags = (int2*)w.keys;                      // the unsorted keys are dead once sorted
  w.scan = (int2*)p; p += align_up(nc * 8);
  w.part_loss = (double*)p; p += align_up((size_t)ROW_CTAS_MAX * 8);
  w.part_cnt = (long long*)p; p += align_up((size_t)ROW_CTAS_MAX * 16);
  w.part_ap = (double*)p; p += align_up((size_t)C * ap_chunks(n) * 8);
  w.cub = p; w.cub_bytes = cub_bytes(n, C);
  return w;
}

}  // namespace

extern "C" size_t pcb_seg_eval_ws_bytes(int64_t n, int C) {
  if (n < 1) n = 1;
  if (C < 2) C = 2;
  if (C > 64) C = 64;
  const size_t nc = (size_t)n * C;
  return 3 * align_up(nc * 8) + align_up((size_t)ROW_CTAS_MAX * 8) + align_up((size_t)ROW_CTAS_MAX * 16) +
         align_up((size_t)C * ap_chunks(n) * 8) + align_up(cub_bytes(n, C));
}

extern "C" int pcb_seg_eval(const float* logits, const int64_t* target, int64_t n, int C, int64_t ignore_index, int32_t* pred, int64_t* hist,
                            double* stats, double* ap, float* prob, void* ws, size_t ws_bytes, void* stream) {
  PCB_ARG(C >= 2 && C <= 64 && n >= 1 && n * C < (1ll << 31));
  PCB_ARG(logits && target && hist && stats && ap && ws);
  PCB_ARG(ws_bytes >= pcb_seg_eval_ws_bytes(n, C));
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t total = n * C;
  Ws w = carve(ws, n, C);
  const int g_rows = row_ctas(n);
  const size_t smem = rows_smem(C);
  PCB_CUDA(cudaFuncSetAttribute(seg_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  launch_kernel(seg_rows_kernel, g_rows, ROWS, smem, st, logits, target, n, C, ignore_index, pred, prob, w.keys,
                (unsigned long long*)hist, w.part_loss, w.part_cnt);
  if (int e = check_launch("seg_rows_kernel")) return e;
  size_t cb = w.cub_bytes;
  PCB_CUDA(cub::DeviceRadixSort::SortKeys(w.cub, cb, (const uint64_t*)w.keys, w.sorted, (int)total, 0, key_bits(C), st));
  launch_kernel(ap_flags_kernel, (unsigned)((total + 255) / 256), 256, 0, st, (const uint64_t*)w.sorted, n, total, w.flags);
  if (int e = check_launch("ap_flags_kernel")) return e;
  cb = w.cub_bytes;
  PCB_CUDA(cub::DeviceScan::InclusiveScan(w.cub, cb, (const int2*)w.flags, w.scan, SumMax(), (int)total, st));
  const int chunks = ap_chunks(n);
  launch_kernel(ap_terms_kernel, dim3(chunks, C), AP_THREADS, 0, st, (const uint64_t*)w.sorted, (const int2*)w.scan, n, w.part_ap);
  if (int e = check_launch("ap_terms_kernel")) return e;
  launch_kernel(seg_final_kernel, 1, 256, 0, st, (const double*)w.part_loss, (const long long*)w.part_cnt, g_rows, (const double*)w.part_ap,
                chunks, (const int2*)w.scan, n, C, stats, ap);
  g_launches.fetch_add(8);                                 // the sort's and the scan's kernels
  return check_launch("seg_final_kernel");
}
