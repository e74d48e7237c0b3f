// Contrastive-loss kernels and the flat-buffer SGD step.
//   PointInfoNCE: logits = q k^T / T, softmax cross-entropy against the diagonal, and its gradients
//   (replaces torch.mm + nn.CrossEntropyLoss, pretrain/pointcontrast/lib/ddp_trainer.py:420-426, lib/criterion.py:15-19).
//   Hardest-contrastive: fused pairwise distance + row min/argmin (replaces the 537 MB broadcast `pdist`
//   + .min(1), lib/ddp_trainer.py:182-184,215-219).
// These are < 1 % of a training step; they are exact-fp32 SIMT kernels.
#include <stdlib.h>
#include "common.cuh"

using namespace pcb;

namespace {

// C[M,N] = alpha * op(A) op(B).  TA: A stored [K,M] (else [M,K]);  TB: B stored [N,K] (else [K,N]).  Row-major, fp32.
template <bool TA, bool TB>
__global__ void __launch_bounds__(256) sgemm_kernel(const float* __restrict__ A, int lda, const float* __restrict__ B, int ldb,
                                                    float* __restrict__ C, int ldc, int M, int N, int K, float alpha) {
  __shared__ float As[16][68];
  __shared__ float Bs[16][68];
  const int t = threadIdx.x;
  const int tx = t & 15, ty = t >> 4;          // 16 x 16 threads, 4 x 4 outputs each
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += 16) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int m, k;
      if (TA) { m = t & 63; k = (t >> 6) + 4 * i; } else { k = t & 15; m = (t >> 4) + 16 * i; }
      float v = 0.f;
      if (m0 + m < M && k0 + k < K) v = TA ? A[(int64_t)(k0 + k) * lda + m0 + m] : A[(int64_t)(m0 + m) * lda + k0 + k];
      As[k][m] = v;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int n, k;
      if (TB) { k = t & 15; n = (t >> 4) + 16 * i; } else { n = t & 63; k = (t >> 6) + 4 * i; }
      float v = 0.f;
      if (n0 + n < N && k0 + k < K) v = TB ? B[(int64_t)(n0 + n) * ldb + k0 + k] : B[(int64_t)(k0 + k) * ldb + n0 + n];
      Bs[k][n] = v;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[k][ty * 4 + i]; b[i] = Bs[k][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int m = m0 + ty * 4 + i, n = n0 + tx * 4 + j;
      if (m < M && n < N) C[(int64_t)m * ldc + n] = alpha * acc[i][j];
    }
}

// one CTA per row: lse, row loss, and in-place gradient  G[i][j] = (softmax_ij - delta_ij) * scale
__global__ void nce_softmax_kernel(float* __restrict__ L, int64_t n, float scale, float* __restrict__ rowloss) {
  __shared__ float red[32];
  const int64_t i = blockIdx.x;
  float* row = L + i * n;
  const int t = threadIdx.x, lane = t & 31, w = t >> 5, nw = blockDim.x >> 5;
  float m = -INFINITY;
  for (int64_t j = t; j < n; j += blockDim.x) m = fmaxf(m, row[j]);
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (lane == 0) red[w] = m;
  __syncthreads();
  m = red[0];
  for (int k = 1; k < nw; ++k) m = fmaxf(m, red[k]);
  __syncthreads();
  float s = 0.f;
  for (int64_t j = t; j < n; j += blockDim.x) s += expf(row[j] - m);
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) red[w] = s;
  __syncthreads();
  s = 0.f;
  for (int k = 0; k < nw; ++k) s += red[k];
  const float lse = m + logf(s);
  const float diag = row[i];
  __syncthreads();
  for (int64_t j = t; j < n; j += blockDim.x) {
    float p = expf(row[j] - lse);
    row[j] = (p - (j == i ? 1.f : 0.f)) * scale;
  }
  if (t == 0) rowloss[i] = lse - diag;
}

__global__ void mean_kernel(const float* __restrict__ v, int64_t n, float* __restrict__ out) {
  __shared__ double red[32];
  double s = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) s += (double)v[i];
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tot = 0.0;
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) tot += red[k];
    *out = (float)(tot / (double)n);
  }
}

// packed[i] = min over j of (bits(d2_ij) << 32 | j)
__global__ void __launch_bounds__(256) pdist_min_kernel(const float* __restrict__ A, int64_t P, const float* __restrict__ B,
                                                        int64_t S, int D, int s_per_split, unsigned long long* packed) {
  extern __shared__ float sm[];
  float* As = sm;                       // [64][D+1]
  float* Bs = sm + 64 * (D + 1);        // [64][D]
  const int t = threadIdx.x;
  const int il = t & 63, jl = t >> 6;
  const int64_t i0 = (int64_t)blockIdx.x * 64;
  for (int e = t; e < 64 * D; e += 256) {
    int r = e / D, d = e - r * D;
    As[r * (D + 1) + d] = (i0 + r < P) ? A[(i0 + r) * D + d] : 0.f;
  }
  const int64_t j_begin = (int64_t)blockIdx.y * s_per_split;
  const int64_t j_end = min(S, j_begin + s_per_split);
  unsigned long long best = ~0ull;
  for (int64_t j0 = j_begin; j0 < j_end; j0 += 64) {
    __syncthreads();
    for (int e = t; e < 64 * D; e += 256) {
      int r = e / D, d = e - r * D;
      Bs[e] = (j0 + r < j_end) ? B[(j0 + r) * D + d] : 0.f;
    }
    __syncthreads();
    const float* a = As + il * (D + 1);
    for (int jj = jl; jj < 64; jj += 4) {
      if (j0 + jj >= j_end) break;
      const float* b = Bs + jj * D;
      float d2 = 0.f;
      for (int d = 0; d < D; ++d) { float df = a[d] - b[d]; d2 = fmaf(df, df, d2); }
      unsigned long long pk = ((unsigned long long)__float_as_uint(d2) << 32) | (unsigned long long)(uint32_t)(j0 + jj);
      best = pk < best ? pk : best;
    }
  }
  if (i0 + il < P && best != ~0ull) atomicMin(packed + i0 + il, best);
}

__global__ void pdist_unpack_kernel(const unsigned long long* __restrict__ packed, int64_t P, float* __restrict__ minval,
                                    int32_t* __restrict__ argmin) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= P) return;
  unsigned long long pk = packed[i];
  minval[i] = sqrtf(__uint_as_float((uint32_t)(pk >> 32)) + 1e-7f);
  argmin[i] = (int32_t)(pk & 0xFFFFFFFFull);
}

__global__ void sgd_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ buf, int64_t n, float lr,
                           float momentum, float wd, float gscale, int first, float keep) {
  pdl_wait(); pdl_trigger();
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int64_t n4 = n >> 2;
  if (i < n4) {
    float4 P = reinterpret_cast<float4*>(p)[i];
    float4 G = __ldg(reinterpret_cast<const float4*>(g) + i);
    float4 Bf = first ? make_float4(0, 0, 0, 0) : reinterpret_cast<float4*>(buf)[i];
    float4 d = make_float4(G.x * gscale + wd * P.x, G.y * gscale + wd * P.y, G.z * gscale + wd * P.z, G.w * gscale + wd * P.w);
    if (first) Bf = d;
    else { Bf.x = momentum * Bf.x + keep * d.x; Bf.y = momentum * Bf.y + keep * d.y; Bf.z = momentum * Bf.z + keep * d.z; Bf.w = momentum * Bf.w + keep * d.w; }
    P.x -= lr * Bf.x; P.y -= lr * Bf.y; P.z -= lr * Bf.z; P.w -= lr * Bf.w;
    reinterpret_cast<float4*>(buf)[i] = Bf;
    reinterpret_cast<float4*>(p)[i] = P;
  } else {
    int64_t e = (n4 << 2) + (i - n4);
    if (e < n) {
      float d = g[e] * gscale + wd * p[e];
      float b = first ? d : momentum * buf[e] + keep * d;
      buf[e] = b;
      p[e] -= lr * b;
    }
  }
}

template <bool TA, bool TB>
int launch_sgemm(const float* A, int lda, const float* B, int ldb, float* C, int ldc, int M, int N, int K, float alpha,
                 cudaStream_t st) {
  dim3 grid((N + 63) / 64, (M + 63) / 64);
  sgemm_kernel<TA, TB><<<grid, 256, 0, st>>>(A, lda, B, ldb, C, ldc, M, N, K, alpha);
  return check_launch("sgemm_kernel");
}

}  // namespace

namespace pcb {
bool nce_tc_supported(int64_t n, int D);
size_t nce_tc_ws_bytes(int64_t n, int D);
int nce_tc_forward_backward(const float* q, const float* k, int64_t n, int D, float inv_T, float* loss, float* dq, float* dk, void* ws,
                            cudaStream_t st);
}

// scratch: the tensor-core path needs O(n * D) (partial statistics / gradients); the exact-fp32 SIMT path (feature widths other
// than 32 / 64, or PCB_NCE_SIMT=1) materialises the n x n logits
extern "C" size_t pcb_nce_ws_bytes(int64_t n) {
  size_t simt = (size_t)n * n * sizeof(float) + (size_t)n * sizeof(float) + 512, tc = nce_tc_ws_bytes(n, 64);
  return simt > tc ? simt : tc;
}

extern "C" int pcb_nce_forward_backward(const float* q, const float* k, int64_t n, int D, float inv_T, float* loss, float* dq,
                                        float* dk, void* ws, size_t ws_bytes, void* stream) {
  PCB_ARG(q && k && loss && dq && dk && ws && n >= 1 && n <= 46000 && D >= 1);
  PCB_ARG(ws_bytes >= pcb_nce_ws_bytes(n) - 512);
  cudaStream_t st = (cudaStream_t)stream;
  static int force_simt = -1;
  if (force_simt < 0) { const char* e = getenv("PCB_NCE_SIMT"); force_simt = (e && atoi(e)) ? 1 : 0; }
  ProfScope prof(st, 4);
  if (!force_simt && nce_tc_supported(n, D)) return nce_tc_forward_backward(q, k, n, D, inv_T, loss, dq, dk, ws, st);
  float* L = (float*)ws;
  float* rowloss = L + n * n;
  if (int e = launch_sgemm<false, true>(q, D, k, D, L, (int)n, (int)n, (int)n, D, inv_T, st)) return e;
  nce_softmax_kernel<<<(unsigned)n, 256, 0, st>>>(L, n, inv_T / (float)n, rowloss);
  if (int e = check_launch("nce_softmax_kernel")) return e;
  mean_kernel<<<1, 1024, 0, st>>>(rowloss, n, loss);
  if (int e = check_launch("mean_kernel")) return e;
  if (int e = launch_sgemm<false, false>(L, (int)n, k, D, dq, D, (int)n, D, (int)n, 1.f, st)) return e;    // dq = G k
  return launch_sgemm<true, false>(L, (int)n, q, D, dk, D, (int)n, D, (int)n, 1.f, st);                     // dk = G^T q
}

// ------------------------------------------------------------------------------------------------ L2 normalisation of feature rows
// y = x / ||x||_2 per row, no epsilon (`model/res16unet.py:262-266`); one warp per row, lanes stride over the channels.
namespace {
__global__ void l2norm_fwd_kernel(const float* __restrict__ X, int64_t n, int C, float* __restrict__ Y, float* __restrict__ inv_norm) {
  pdl_wait(); pdl_trigger();
  const int lane = threadIdx.x & 31;
  const int64_t row = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n) return;
  float ss = 0.f;
  for (int c = lane; c < C; c += 32) { const float v = X[row * C + c]; ss = fmaf(v, v, ss); }
  for (int o = 16; o; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const float inv = 1.0f / sqrtf(ss);
  for (int c = lane; c < C; c += 32) Y[row * C + c] = X[row * C + c] * inv;
  if (lane == 0) inv_norm[row] = inv;
}
// dx = (dy - y (y . dy)) / ||x||
__global__ void l2norm_bwd_kernel(const float* __restrict__ dY, const float* __restrict__ Y, const float* __restrict__ inv_norm, int64_t n,
                                  int C, float* __restrict__ dX) {
  pdl_wait(); pdl_trigger();
  const int lane = threadIdx.x & 31;
  const int64_t row = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n) return;
  float dot = 0.f;
  for (int c = lane; c < C; c += 32) dot = fmaf(Y[row * C + c], dY[row * C + c], dot);
  for (int o = 16; o; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
  const float inv = inv_norm[row];
  for (int c = lane; c < C; c += 32) dX[row * C + c] = (dY[row * C + c] - Y[row * C + c] * dot) * inv;
}
}  // namespace

extern "C" int pcb_l2norm_forward(const float* X, int64_t n, int C, float* Y, float* inv_norm, void* stream) {
  PCB_ARG(n >= 0 && C >= 1);
  if (n == 0) return PCB_OK;
  PCB_ARG(X && Y && inv_norm);
  launch_kernel(l2norm_fwd_kernel, (unsigned)((n + 7) / 8), 256, 0, (cudaStream_t)stream, X, n, C, Y, inv_norm);
  return check_launch("l2norm_fwd_kernel");
}

extern "C" int pcb_l2norm_backward(const float* dY, const float* Y, const float* inv_norm, int64_t n, int C, float* dX, void* stream) {
  PCB_ARG(n >= 0 && C >= 1);
  if (n == 0) return PCB_OK;
  PCB_ARG(dY && Y && inv_norm && dX);
  launch_kernel(l2norm_bwd_kernel, (unsigned)((n + 7) / 8), 256, 0, (cudaStream_t)stream, dY, Y, inv_norm, n, C, dX);
  return check_launch("l2norm_bwd_kernel");
}

extern "C" int pcb_pdist_rowmin(const float* A, int64_t P, const float* B, int64_t S, int D, float* minval, int32_t* argmin,
                                uint64_t* packed, void* stream) {
  PCB_ARG(A && B && minval && argmin && packed && P >= 1 && S >= 1 && D >= 1 && D <= 64);
  cudaStream_t st = (cudaStream_t)stream;
  PCB_CUDA(cudaMemsetAsync(packed, 0xFF, (size_t)P * sizeof(uint64_t), st));
  int rowblocks = (int)((P + 63) / 64);
  int splits = (2 * num_sms() + rowblocks - 1) / rowblocks;
  int max_splits = (int)((S + 63) / 64);
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  int sps = (int)((S + splits - 1) / splits);
  sps = (sps + 63) / 64 * 64;
  splits = (int)((S + sps - 1) / sps);
  size_t smem = (size_t)(64 * (D + 1) + 64 * D) * sizeof(float);
  dim3 grid(rowblocks, splits);
  pdist_min_kernel<<<grid, 256, smem, st>>>(A, P, B, S, D, sps, (unsigned long long*)packed);
  if (int e = check_launch("pdist_min_kernel")) return e;
  pdist_unpack_kernel<<<(unsigned)((P + 255) / 256), 256, 0, st>>>((const unsigned long long*)packed, P, minval, argmin);
  return check_launch("pdist_unpack_kernel");
}

// ------------------------------------------------------------------------------------------------ cross-entropy (semantic segmentation)
// nn.CrossEntropyLoss(ignore_index) over logits [n, C] (`downstream/semseg/lib/train.py:68,120`): loss = mean over the rows whose
// target != ignore of (logsumexp(x) - x[target]); dlogits = (softmax(x) - onehot) * scale / count on those rows, 0 elsewhere.
// One warp per row (C <= 1024), two passes: per-row loss + validity, then the mean, then the gradient.
namespace {
__global__ void ce_rows_kernel(const float* __restrict__ X, const int64_t* __restrict__ target, int64_t n, int C, int64_t ignore,
                               float* __restrict__ rowloss, float* __restrict__ rowlse) {
  pdl_wait(); pdl_trigger();
  const int lane = threadIdx.x & 31;
  const int64_t row = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n) return;
  const int64_t t = target[row];
  float m, s;
  const float lse = row_logsumexp<32>(X + row * C, C, lane, m, s);
  if (lane == 0) {
    rowlse[row] = lse;
    rowloss[row] = (t == ignore || t < 0 || t >= C) ? 0.f : lse - X[row * C + t];
  }
}
// out[0] = sum(rowloss) / count, out[1] = count   (count = rows with a valid target; fp64, fixed order)
__global__ void ce_mean_kernel(const float* __restrict__ rowloss, const int64_t* __restrict__ target, int64_t n, int C, int64_t ignore,
                               float* __restrict__ out) {
  pdl_wait(); pdl_trigger();
  __shared__ double s_sum[32];
  __shared__ double s_cnt[32];
  double s = 0.0, cnt = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    const int64_t t = target[i];
    if (!(t == ignore || t < 0 || t >= C)) { s += rowloss[i]; cnt += 1.0; }
  }
  for (int o = 16; o; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); cnt += __shfl_xor_sync(0xffffffffu, cnt, o); }
  if ((threadIdx.x & 31) == 0) { s_sum[threadIdx.x >> 5] = s; s_cnt[threadIdx.x >> 5] = cnt; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double ts = 0.0, tc = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { ts += s_sum[w]; tc += s_cnt[w]; }
    out[0] = (float)(ts / tc);       // 0/0 = nan when every row is ignored, as torch
    out[1] = (float)tc;
  }
}
__global__ void ce_grad_kernel(const float* __restrict__ X, const int64_t* __restrict__ target, const float* __restrict__ rowlse,
                               const float* __restrict__ stats, int64_t n, int C, int64_t ignore, float scale, float* __restrict__ dX) {
  pdl_wait(); pdl_trigger();
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= n * C) return;
  const int64_t row = e / C;
  const int c = (int)(e - row * C);
  const int64_t t = target[row];
  float g = 0.f;
  if (!(t == ignore || t < 0 || t >= C)) g = (expf(X[e] - rowlse[row]) - (c == t ? 1.f : 0.f)) * (scale / stats[1]);
  dX[e] = g;
}
}  // namespace

extern "C" size_t pcb_ce_ws_bytes(int64_t n) { return (size_t)(2 * n + 4) * sizeof(float) + 256; }

extern "C" int pcb_ce_forward_backward(const float* logits, const int64_t* target, int64_t n, int C, int64_t ignore_index, float grad_scale,
                                       float* loss, float* dlogits, void* ws, size_t ws_bytes, void* stream) {
  PCB_ARG(logits && target && loss && dlogits && ws && n >= 1 && C >= 1 && C <= 1024 && ws_bytes >= pcb_ce_ws_bytes(n) - 256);
  cudaStream_t st = (cudaStream_t)stream;
  float* rowloss = (float*)ws;
  float* rowlse = rowloss + n;
  float* stats = rowlse + n;
  launch_kernel(ce_rows_kernel, (unsigned)((n + 7) / 8), 256, 0, st, logits, target, n, C, ignore_index, rowloss, rowlse);
  if (int e = check_launch("ce_rows_kernel")) return e;
  launch_kernel(ce_mean_kernel, 1, 1024, 0, st, (const float*)rowloss, target, n, C, ignore_index, stats);
  if (int e = check_launch("ce_mean_kernel")) return e;
  PCB_CUDA(cudaMemcpyAsync(loss, stats, sizeof(float), cudaMemcpyDeviceToDevice, st));
  launch_kernel(ce_grad_kernel, (unsigned)((n * C + 255) / 256), 256, 0, st, logits, target, (const float*)rowlse, (const float*)stats, n, C,
                ignore_index, grad_scale, dlogits);
  return check_launch("ce_grad_kernel");
}

extern "C" int pcb_sgd_step(float* p, const float* g, float* buf, int64_t n, float lr, float momentum, float weight_decay,
                            float grad_scale, int first, float dampening, void* stream) {
  PCB_ARG(n >= 0);
  if (n == 0) return PCB_OK;
  PCB_ARG(p && g && buf);
  ProfScope prof((cudaStream_t)stream, 5);
  int64_t threads = (n >> 2) + (n & 3);
  launch_kernel(sgd_kernel, (unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream, p, g, buf, n, lr, momentum, weight_decay,
                grad_scale, first, 1.0f - dampening);
  return check_launch("sgd_kernel");
}
