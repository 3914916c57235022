// Training-side kernels (SURVEY.md §8 row A15 / BASELINE config 4): everything the backward pass of
// TouchedRegraster.training_step (model5_b.py:912-1155) needs that the inference library does not have.
//   * pz_sgemm          generic fp32 GEMM with arbitrary operand strides (NN/NT/TN/TT), batching, split-K and a
//                       bias / ReLU / ReLU-mask epilogue -- dX = dY W, dW = dY^T X, the attention GEMMs and the
//                       train-mode forward layers all go through it (FFMA pipe; fp32 like the reference, no AMP)
//   * pz_colsum         bias gradients
//   * pz_bn_point_*     nn.BatchNorm1d(1024) over the POINT index in train mode (model5_b.py:424-425, :447-448)
//   * pz_maxpool_*      neighbourhood / point max-pool with arg-max and its scatter backward
//   * pz_scatter_add_rows   backward of index_points (pointnet_util.py:39-50)
//   * pz_softmax_bwd    backward of scaled_dot_production's softmax (model5_b.py:67-75)
//   * pz_cross_entropy  F.cross_entropy(logits [B,2,N], target [B,N]) forward + backward (model5_b.py:1063-1064)
//   * pz_pose_grad      d loss / d twist through se3.exp + se3.transform (+ comp) (model5_b.py:947-967)
//   * pz_se3_exp_backward, pz_comp_backward   the autograd backward of se3.exp and of comp on their own
//   * pz_adam_step      torch.optim.Adam on one flat parameter buffer (model5_b.py:1453-1457)
#include <math.h>

#include "pz_common.cuh"

namespace pz {
namespace {

// =============================================================================== generic SGEMM
// C[m,n] (+)= alpha * sum_k A(m,k) B(k,n);  A(m,k) = A[m*sam + k*sak], B(k,n) = B[k*sbk + n*sbn].
// 128x128x8 tiles, 256 threads, 8x8 micro-tiles, register prefetch of the next tile.
struct SgemmArgs {
  const float *A, *B;
  float* C;
  long long sam, sak, sbk, sbn, ldc;
  long long bsa, bsb, bsc;   // batch strides (blockIdx.z = batch when splitk == 1)
  int M, N, K;
  int splitk;                // >1: blockIdx.z = K split, partial sums are atomically added into C
  float alpha, beta;
  const float* bias;         // [N] added after alpha*acc
  int relu;
  const float* mask;         // epilogue multiplies by (mask[m*ldmask + n] > 0)
  long long ldmask, bsmask;
  const float* residual;     // added last: C = residual + f(acc)
  long long ldres, bsres;
};

constexpr int GK = 8;

// GT x GT output tile (128: 8x8 micro-tiles; 64: 4x4, for outputs no wider than 64 -- the weight gradients of the
// 64-channel layers, where a 128-wide tile would be 3/4 empty), GK-deep k-steps, 256 threads.
template <bool A_KCONTIG, bool B_NCONTIG, int GT>
__global__ void __launch_bounds__(256) sgemm_kernel(const SgemmArgs p) {
  constexpr int MT = GT / 16;            // micro-tile edge per thread
  constexpr int EPT = GT * GK / 256;     // operand elements each thread loads per k-step (4 or 2)
  __shared__ __align__(16) float As[2][GK][GT + 4];
  __shared__ __align__(16) float Bs[2][GK][GT + 4];
  const int t = threadIdx.x;
  const int m0 = blockIdx.y * GT, n0 = blockIdx.x * GT;
  int kbeg = 0, kend = p.K;
  const float *A = p.A, *B = p.B;
  float* C = p.C;
  const float* mask = p.mask;
  const float* residual = p.residual;
  if (p.splitk > 1) {
    const int chunk = ((p.K + p.splitk - 1) / p.splitk + GK - 1) / GK * GK;
    kbeg = blockIdx.z * chunk;
    kend = min(p.K, kbeg + chunk);
    if (kbeg >= kend) return;
  } else {
    A += (long long)blockIdx.z * p.bsa;
    B += (long long)blockIdx.z * p.bsb;
    C += (long long)blockIdx.z * p.bsc;
    if (mask) mask += (long long)blockIdx.z * p.bsmask;
    if (residual) residual += (long long)blockIdx.z * p.bsres;
  }
  // loader coordinates: EPT consecutive elements (along the contiguous dimension) per thread per operand
  constexpr int KT = GK / EPT;           // threads along k when k is contiguous
  constexpr int MTH = GT / EPT;          // threads along m / n when that dimension is contiguous
  int a_m, a_k, b_k, b_n;
  if (A_KCONTIG) { a_m = t / KT; a_k = (t % KT) * EPT; } else { a_k = t / MTH; a_m = (t % MTH) * EPT; }
  if (B_NCONTIG) { b_k = t / MTH; b_n = (t % MTH) * EPT; } else { b_n = t / KT; b_k = (t % KT) * EPT; }
  float ra[EPT], rb[EPT];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int i = 0; i < EPT; ++i) {
      const int m = m0 + a_m + (A_KCONTIG ? 0 : i), k = k0 + a_k + (A_KCONTIG ? i : 0);
      ra[i] = (m < p.M && k < kend) ? A[(long long)m * p.sam + (long long)k * p.sak] : 0.f;
      const int kk = k0 + b_k + (B_NCONTIG ? 0 : i), n = n0 + b_n + (B_NCONTIG ? i : 0);
      rb[i] = (kk < kend && n < p.N) ? B[(long long)kk * p.sbk + (long long)n * p.sbn] : 0.f;
    }
  };
  auto stash = [&](int buf) {
#pragma unroll
    for (int i = 0; i < EPT; ++i) {
      if (A_KCONTIG) As[buf][a_k + i][a_m] = ra[i]; else As[buf][a_k][a_m + i] = ra[i];
      if (B_NCONTIG) Bs[buf][b_k][b_n + i] = rb[i]; else Bs[buf][b_k + i][b_n] = rb[i];
    }
  };
  float acc[MT][MT];
#pragma unroll
  for (int i = 0; i < MT; ++i)
#pragma unroll
    for (int j = 0; j < MT; ++j) acc[i][j] = 0.f;
  const int ty = t >> 4, tx = t & 15;
  fetch(kbeg);
  stash(0);
  __syncthreads();
  int buf = 0;
  for (int k0 = kbeg; k0 < kend; k0 += GK) {
    const bool more = k0 + GK < kend;
    if (more) fetch(k0 + GK);
#pragma unroll
    for (int kk = 0; kk < GK; ++kk) {
      float a[MT], b[MT];
      // rows ty*4+{0..3} (and GT/2 + the same for the 8x8 micro-tile); likewise columns from tx
#pragma unroll
      for (int h = 0; h < MT / 4; ++h) {
        const float4 a4 = *reinterpret_cast<const float4*>(&As[buf][kk][h * (GT / 2) + ty * 4]);
        const float4 b4 = *reinterpret_cast<const float4*>(&Bs[buf][kk][h * (GT / 2) + tx * 4]);
        a[h * 4] = a4.x; a[h * 4 + 1] = a4.y; a[h * 4 + 2] = a4.z; a[h * 4 + 3] = a4.w;
        b[h * 4] = b4.x; b[h * 4 + 1] = b4.y; b[h * 4 + 2] = b4.z; b[h * 4 + 3] = b4.w;
      }
#pragma unroll
      for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < MT; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (more) {
      stash(buf ^ 1);
      __syncthreads();
      buf ^= 1;
    }
  }
#pragma unroll
  for (int i = 0; i < MT; ++i) {
    const int m = m0 + (i >> 2) * (GT / 2) + ty * 4 + (i & 3);
    if (m >= p.M) continue;
#pragma unroll
    for (int j = 0; j < MT; ++j) {
      const int n = n0 + (j >> 2) * (GT / 2) + tx * 4 + (j & 3);
      if (n >= p.N) continue;
      float v = p.alpha * acc[i][j];
      float* c = C + (long long)m * p.ldc + n;
      if (p.splitk > 1) {
        atomicAdd(c, v);
        continue;
      }
      if (p.bias) v += p.bias[n];
      if (p.beta != 0.f) v += p.beta * *c;
      if (p.relu) v = fmaxf(v, 0.f);
      if (mask) v = mask[(long long)m * p.ldmask + n] > 0.f ? v : 0.f;
      if (residual) v += residual[(long long)m * p.ldres + n];
      *c = v;
    }
  }
}

template <int GT>
static void sgemm_dispatch(const SgemmArgs& p, int transA, int transB, int batch_or_splits, cudaStream_t st) {
  dim3 grid((p.N + GT - 1) / GT, (p.M + GT - 1) / GT, batch_or_splits);
  if (!transA && !transB) sgemm_kernel<true, true, GT><<<grid, 256, 0, st>>>(p);
  else if (!transA && transB) sgemm_kernel<true, false, GT><<<grid, 256, 0, st>>>(p);
  else if (transA && !transB) sgemm_kernel<false, true, GT><<<grid, 256, 0, st>>>(p);
  else sgemm_kernel<false, false, GT><<<grid, 256, 0, st>>>(p);
}

// =============================================================================== small helpers
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ x, long long ld, long long M, int N,
                                                     long long rows_per_cta, float* __restrict__ out) {
  // CTA (x, y): 32 columns x one chunk of rows; 8 row-lanes, tree over the lanes, one atomicAdd per column
  __shared__ float red[8][33];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31), r0 = threadIdx.x >> 5;
  const long long rb = (long long)blockIdx.y * rows_per_cta, re = min(M, rb + rows_per_cta);
  float acc = 0.f;
  if (c < N)
    for (long long r = rb + r0; r < re; r += 8) acc += x[r * ld + c];
  red[r0][threadIdx.x & 31] = acc;
  __syncthreads();
  if (threadIdx.x < 32 && c < N) {
    float s = 0.f;
    for (int i = 0; i < 8; ++i) s += red[i][threadIdx.x];
    atomicAdd(out + c, s);
  }
}

__global__ void __launch_bounds__(256) scale_kernel(float* __restrict__ x, int n, float a) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < n) x[i] = a == 0.f ? 0.f : a * x[i];
}

__global__ void __launch_bounds__(256) axpby_kernel(long long n, float a, const float* __restrict__ x, float b,
                                                    const float* __restrict__ y, float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
  if (i < n) out[i] = a * x[i] + (y ? b * y[i] : 0.f);
}

// x[r*ld + c] = act(x[r*ld + c] + bias[c])  (finishes a split-K forward GEMM)
__global__ void __launch_bounds__(256) bias_act_kernel(long long rows, int cols, float* __restrict__ x, long long ld,
                                                       const float* __restrict__ bias, int relu) {
  const long long e = (long long)blockIdx.x * 256 + threadIdx.x;
  if (e >= rows * cols) return;
  const long long r = e / cols;
  const int c = (int)(e - r * cols);
  float v = x[r * ld + c] + (bias ? bias[c] : 0.f);
  x[r * ld + c] = relu ? fmaxf(v, 0.f) : v;
}

// strided 2-D variant: out[r*ldo + c] = a*x[r*ldx + c] + b*y[r*ldy + c]
__global__ void __launch_bounds__(256) axpby2d_kernel(long long rows, int cols, float a, const float* __restrict__ x,
                                                      long long ldx, float b, const float* __restrict__ y, long long ldy,
                                                      float* __restrict__ out, long long ldo) {
  const long long e = (long long)blockIdx.x * 256 + threadIdx.x;
  if (e >= rows * cols) return;
  const long long r = e / cols;
  const int c = (int)(e - r * cols);
  out[r * ldo + c] = a * x[r * ldx + c] + (y ? b * y[r * ldy + c] : 0.f);
}

// out = mask > 0 ? dy : 0   (the ReLU gate applied to an incoming gradient)
__global__ void __launch_bounds__(256) relu_gate_kernel(long long rows, int cols, const float* __restrict__ dy,
                                                        long long ldy, const float* __restrict__ mask, long long ldm,
                                                        float* __restrict__ out, long long ldo) {
  const long long e = (long long)blockIdx.x * 256 + threadIdx.x;
  if (e >= rows * cols) return;
  const long long r = e / cols;
  const int c = (int)(e - r * cols);
  out[r * ldo + c] = mask[r * ldm + c] > 0.f ? dy[r * ldy + c] : 0.f;
}

// dst[(g*reps + r)*ldd + c] = src[g*C + c]   (x.repeat(1, reps, 1) of a per-cloud row, model5_b.py:742)
__global__ void __launch_bounds__(256) broadcast_rows_kernel(const float* __restrict__ src, long long G, int reps, int C,
                                                             float* __restrict__ dst, long long ldd) {
  const long long e = (long long)blockIdx.x * 256 + threadIdx.x;
  if (e >= G * reps * C) return;
  const int c = (int)(e % C);
  const long long row = e / C;
  dst[row * ldd + c] = src[(row / reps) * C + c];
}

// y[g, c] = sum_k x[(g*K + k)*ld + c]   (backward of the broadcast above); one warp-row per (g, 32 columns)
__global__ void __launch_bounds__(256) group_sum_kernel(const float* __restrict__ x, long long ld, long long G, int K,
                                                        int C, float* __restrict__ y) {
  __shared__ float red[8][33];
  const long long g = blockIdx.y;
  const int c = blockIdx.x * 32 + (threadIdx.x & 31), r0 = threadIdx.x >> 5;
  float acc = 0.f;
  if (c < C)
    for (int k = r0; k < K; k += 8) acc += x[(g * K + k) * ld + c];
  red[r0][threadIdx.x & 31] = acc;
  __syncthreads();
  if (threadIdx.x < 32 && c < C) {
    float s = 0.f;
    for (int i = 0; i < 8; ++i) s += red[i][threadIdx.x];
    y[g * C + c] = s;
  }
}

// =============================================================================== BatchNorm over the point index
// x [B, P, C]: statistics per point p over the B*C values (train mode).  grid = P, block = 256.
__device__ __forceinline__ float block_sum_256(float v, float* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = 0.f;
  if (threadIdx.x < 8) r = red[threadIdx.x];
  if (threadIdx.x < 32)
    for (int o = 4; o > 0; o >>= 1) r += __shfl_down_sync(0xffffffffu, r, o);
  if (threadIdx.x == 0) red[8] = r;
  __syncthreads();
  return red[8];
}

__global__ void __launch_bounds__(256) bn_point_fwd_kernel(const float* __restrict__ x, int B, int P, int C,
                                                           const float* __restrict__ gamma, const float* __restrict__ beta,
                                                           float* running_mean, float* running_var, float momentum,
                                                           float eps, int relu, float* __restrict__ y,
                                                           float* __restrict__ save_mean, float* __restrict__ save_invstd) {
  __shared__ float red[9];
  const int p = blockIdx.x;
  const int cnt = B * C;
  float s = 0.f;
  for (int e = threadIdx.x; e < cnt; e += 256) s += x[((size_t)(e / C) * P + p) * C + e % C];
  const float mean = block_sum_256(s, red) / (float)cnt;
  float q = 0.f;
  for (int e = threadIdx.x; e < cnt; e += 256) {
    const float d = x[((size_t)(e / C) * P + p) * C + e % C] - mean;
    q = fmaf(d, d, q);
  }
  const float var = block_sum_256(q, red) / (float)cnt;
  const float invstd = rsqrtf(var + eps);
  const float g = gamma[p], bt = beta[p];
  for (int e = threadIdx.x; e < cnt; e += 256) {
    const size_t off = ((size_t)(e / C) * P + p) * C + e % C;
    float v = (x[off] - mean) * invstd * g + bt;
    if (relu) v = fmaxf(v, 0.f);
    y[off] = v;
  }
  if (threadIdx.x == 0) {
    save_mean[p] = mean;
    save_invstd[p] = invstd;
    if (running_mean) {
      const float unbiased = cnt > 1 ? var * (float)cnt / (float)(cnt - 1) : var;
      running_mean[p] = (1.f - momentum) * running_mean[p] + momentum * mean;
      running_var[p] = (1.f - momentum) * running_var[p] + momentum * unbiased;
    }
  }
}

// dy is the gradient w.r.t. the (post-ReLU when relu) output y; dx, dgamma[p], dbeta[p]
__global__ void __launch_bounds__(256) bn_point_bwd_kernel(const float* __restrict__ x, const float* __restrict__ y,
                                                           const float* __restrict__ dy, int B, int P, int C,
                                                           const float* __restrict__ gamma,
                                                           const float* __restrict__ save_mean,
                                                           const float* __restrict__ save_invstd, int relu,
                                                           int accumulate, float* __restrict__ dx,
                                                           float* __restrict__ dgamma, float* __restrict__ dbeta) {
  __shared__ float red[9];
  const int p = blockIdx.x;
  const int cnt = B * C;
  const float mean = save_mean[p], invstd = save_invstd[p], g = gamma[p];
  float sdy = 0.f, sdyx = 0.f;
  for (int e = threadIdx.x; e < cnt; e += 256) {
    const size_t off = ((size_t)(e / C) * P + p) * C + e % C;
    float d = dy[off];
    if (relu && !(y[off] > 0.f)) d = 0.f;
    sdy += d;
    sdyx = fmaf(d, (x[off] - mean) * invstd, sdyx);
  }
  const float db = block_sum_256(sdy, red);
  const float dg = block_sum_256(sdyx, red);
  const float inv_cnt = 1.f / (float)cnt;
  for (int e = threadIdx.x; e < cnt; e += 256) {
    const size_t off = ((size_t)(e / C) * P + p) * C + e % C;
    float d = dy[off];
    if (relu && !(y[off] > 0.f)) d = 0.f;
    const float xh = (x[off] - mean) * invstd;
    dx[off] = g * invstd * (d - db * inv_cnt - xh * dg * inv_cnt);
  }
  if (threadIdx.x == 0) {
    dgamma[p] = accumulate ? dgamma[p] + dg : dg;
    dbeta[p] = accumulate ? dbeta[p] + db : db;
  }
}

// =============================================================================== max-pool with arg-max
// x [G, K, C] -> y [G, C] = max_k, arg [G, C] = first maximising k.  Both directions are pure streaming (the
// backward writes 537 MB per set-abstraction layer at 64 pairs): one CTA per group, every thread owns 4 consecutive
// channels (128-bit accesses) and a subset of the K rows; no per-element index division.
template <int VEC>
__global__ void __launch_bounds__(256) maxpool_fwd_kernel(const float* __restrict__ x, int K, int C,
                                                          float* __restrict__ y, int* __restrict__ arg) {
  const long long g = blockIdx.x;
  const float* px = x + g * (long long)K * C;
  for (int c = threadIdx.x * VEC; c < C; c += blockDim.x * VEC) {      // blockDim = min(256, C / VEC) rounded to a warp
    float best[VEC];
    int bi[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) { best[v] = -INFINITY; bi[v] = 0; }
    for (int k = 0; k < K; ++k) {
      float val[VEC];
      if (VEC == 4) {
        const float4 t = *reinterpret_cast<const float4*>(px + (long long)k * C + c);
        val[0] = t.x; val[1] = t.y; val[2] = t.z; val[3] = t.w;
      } else {
        val[0] = px[(long long)k * C + c];
      }
#pragma unroll
      for (int v = 0; v < VEC; ++v)
        if (val[v] > best[v] || k == 0) { best[v] = val[v]; bi[v] = k; }
    }
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      y[g * C + c + v] = best[v];
      arg[g * C + c + v] = bi[v];
    }
  }
}
// dx [G, K, C] = (k == arg && (!relu_gate || y > 0)) ? dy : 0   (relu_gate: x was a ReLU output, dx is w.r.t. its input)
template <int VEC>
__global__ void __launch_bounds__(256) maxpool_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ y,
                                                          const int* __restrict__ arg, int K, int C, int relu_gate,
                                                          float* __restrict__ dx) {
  const long long g = blockIdx.x;
  const int cols = C / VEC;                       // column groups per row
  const int c = (threadIdx.x % cols) * VEC;       // this thread's channels (cols <= 256 is checked by the launcher
  const int k0 = threadIdx.x / cols;              //  for VEC == 4; the scalar variant loops over column groups)
  const int kstep = 256 / cols;
  if (VEC == 4) {
    if (threadIdx.x >= cols * kstep) return;
    const float4 d4 = *reinterpret_cast<const float4*>(dy + g * C + c);
    const float4 y4 = *reinterpret_cast<const float4*>(y + g * C + c);
    const int4 a4 = *reinterpret_cast<const int4*>(arg + g * C + c);
    const float d[4] = {(!relu_gate || y4.x > 0.f) ? d4.x : 0.f, (!relu_gate || y4.y > 0.f) ? d4.y : 0.f,
                        (!relu_gate || y4.z > 0.f) ? d4.z : 0.f, (!relu_gate || y4.w > 0.f) ? d4.w : 0.f};
    float* px = dx + g * (long long)K * C + c;
    for (int k = k0; k < K; k += kstep)
      *reinterpret_cast<float4*>(px + (long long)k * C) =
          make_float4(a4.x == k ? d[0] : 0.f, a4.y == k ? d[1] : 0.f, a4.z == k ? d[2] : 0.f, a4.w == k ? d[3] : 0.f);
  } else {
    for (int cc = threadIdx.x; cc < C; cc += 256) {
      const long long o = g * C + cc;
      const float d = (!relu_gate || y[o] > 0.f) ? dy[o] : 0.f;
      const int a = arg[o];
      float* px = dx + g * (long long)K * C + cc;
      for (int k = 0; k < K; ++k) px[(long long)k * C] = a == k ? d : 0.f;
    }
  }
}

// =============================================================================== index_points backward
// dst[(m / per_cloud) * N + idx[m], 0:C] += src[m*ld + c0 : c0+C];  one warp per source row (coalesced reads, atomics to
// consecutive addresses), zero entries skipped (the gradient of a max-pooled layer is mostly zeros)
__global__ void __launch_bounds__(256) scatter_add_rows_kernel(const float* __restrict__ src, long long ld, int c0, int C,
                                                               const int64_t* __restrict__ idx, long long M,
                                                               long long per_cloud, int N, float* __restrict__ dst,
                                                               long long ldd) {
  const int lane = threadIdx.x & 31;
  const long long warps = (long long)gridDim.x * 8;
  for (long long m = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); m < M; m += warps) {
    const float* ps = src + m * ld + c0;
    float* pd = dst + ((m / per_cloud) * N + idx[m]) * ldd;
    for (int c = lane; c < C; c += 32) {
      const float v = ps[c];
      if (v != 0.f) atomicAdd(pd + c, v);
    }
  }
}

// =============================================================================== grouped layer 1 without [G*K, 3+D]
// Layer 1 of a grouped MLP splits as  W1 [xyz_j - c_s ; f_j] + b1 = P_j - Q_s  with P (per SOURCE point) and Q (per
// centroid) computed by small GEMMs (DESIGN.md §3); the grouped activation is then a gather:
//   out[r, :] = relu(P[cloud*N + idx[r], :] - Q[r / K, :]),   r = (cloud*S + s)*K + k.   One warp per row.
__global__ void __launch_bounds__(256) gather_sub_relu_kernel(const float* __restrict__ P, const float* __restrict__ Q,
                                                              const int64_t* __restrict__ idx, long long rows, int K,
                                                              int S, int N, int C, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long long warps = (long long)gridDim.x * 8;
  for (long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); r < rows; r += warps) {
    const long long g = r / K;
    const float* p = P + ((g / S) * N + idx[r]) * C;
    const float* q = Q + g * C;
    float* o = out + r * C;
    for (int c = lane * 4; c < C; c += 128) {
      const float4 a = *reinterpret_cast<const float4*>(p + c), b = *reinterpret_cast<const float4*>(q + c);
      *reinterpret_cast<float4*>(o + c) =
          make_float4(fmaxf(a.x - b.x, 0.f), fmaxf(a.y - b.y, 0.f), fmaxf(a.z - b.z, 0.f), fmaxf(a.w - b.w, 0.f));
    }
  }
}
// backward of the gather above for d = gradient w.r.t. the PRE-activation (already ReLU-gated):
//   dP[cloud*N + idx[r], :] += d[r, :] (atomics, zeros skipped),   dQ[g, :] = -sum_k d[g*K + k, :].  One warp per group.
__global__ void __launch_bounds__(256) group_scatter_grad_kernel(const float* __restrict__ d, const int64_t* __restrict__ idx,
                                                                 long long groups, int K, int S, int N, int C,
                                                                 float* __restrict__ dP, float* __restrict__ dQ) {
  const int lane = threadIdx.x & 31;
  const long long warps = (long long)gridDim.x * 8;
  for (long long g = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); g < groups; g += warps) {
    const long long base = (g / S) * N;
    for (int c = lane * 4; c < C; c += 128) {
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int k = 0; k < K; ++k) {
        const long long r = g * K + k;
        const float4 v = *reinterpret_cast<const float4*>(d + r * C + c);
        if (v.x != 0.f || v.y != 0.f || v.z != 0.f || v.w != 0.f) {
          float* t = dP + (base + idx[r]) * C + c;
          if (v.x != 0.f) atomicAdd(t, v.x);
          if (v.y != 0.f) atomicAdd(t + 1, v.y);
          if (v.z != 0.f) atomicAdd(t + 2, v.z);
          if (v.w != 0.f) atomicAdd(t + 3, v.w);
          acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
      }
      *reinterpret_cast<float4*>(dQ + g * C + c) = make_float4(-acc.x, -acc.y, -acc.z, -acc.w);
    }
  }
}

// =============================================================================== softmax forward
// A[r,:] = softmax(scale * S[r,:]);  one warp per row (exp of the shifted logits, as torch.softmax evaluates it)
__global__ void __launch_bounds__(256) softmax_fwd_kernel(const float* __restrict__ S, long long rows, int L, float scale,
                                                          float* __restrict__ A) {
  const long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int lane = threadIdx.x & 31;
  const float* s = S + r * L;
  float mx = -INFINITY;
  for (int j = lane; j < L; j += 32) mx = fmaxf(mx, s[j] * scale);
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float sum = 0.f;
  for (int j = lane; j < L; j += 32) sum += expf(s[j] * scale - mx);
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float inv = 1.f / sum;
  for (int j = lane; j < L; j += 32) A[r * L + j] = expf(s[j] * scale - mx) * inv;
}

// =============================================================================== softmax backward
// dS[r,:] = scale * A[r,:] * (dA[r,:] - sum_j dA[r,j] A[r,j]);  one warp per row
__global__ void __launch_bounds__(256) softmax_bwd_kernel(const float* __restrict__ A, const float* __restrict__ dA,
                                                          long long rows, int L, float scale, float* __restrict__ dS) {
  const long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int lane = threadIdx.x & 31;
  const float* a = A + r * L;
  const float* d = dA + r * L;
  float s = 0.f;
  for (int j = lane; j < L; j += 32) s = fmaf(d[j], a[j], s);
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  for (int j = lane; j < L; j += 32) dS[r * L + j] = scale * a[j] * (d[j] - s);
}

// =============================================================================== cross entropy over 2 classes
// logits [B,2,N], target [B,N] (0/1 as float) -> loss += mean CE ; dlogits = gscale * (softmax - onehot) / (B*N)
__global__ void __launch_bounds__(256) cross_entropy_kernel(const float* __restrict__ logits, const float* __restrict__ target,
                                                            int B, int N, long long sb, long long sc, long long sn,
                                                            float gscale, float* __restrict__ loss,
                                                            float* __restrict__ dlogits) {
  __shared__ float red[9];
  const long long e = (long long)blockIdx.x * 256 + threadIdx.x;
  float li = 0.f;
  if (e < (long long)B * N) {
    const long long b = e / N;
    const int n = (int)(e - b * N);
    const long long o0 = b * sb + n * sn, o1 = o0 + sc;
    const float l0 = logits[o0], l1 = logits[o1];
    const float mx = fmaxf(l0, l1);
    const float e0 = expf(l0 - mx), e1 = expf(l1 - mx);
    const float lse = mx + logf(e0 + e1);
    const int tgt = target[e] != 0.f ? 1 : 0;
    li = lse - (tgt ? l1 : l0);
    if (dlogits) {
      const float inv = gscale / ((float)B * (float)N);
      const float p0 = e0 / (e0 + e1), p1 = e1 / (e0 + e1);
      dlogits[o0] = (p0 - (tgt ? 0.f : 1.f)) * inv;
      dlogits[o1] = (p1 - (tgt ? 1.f : 0.f)) * inv;
    }
  }
  const float s = block_sum_256(li, red);
  if (threadIdx.x == 0) atomicAdd(loss, s / ((float)B * (float)N));
}

// =============================================================================== pose gradient
// forward-mode dual numbers over the 6 twist components: value + d/d(out6)
struct Dual {
  float v, d[6];
};
__device__ __forceinline__ Dual dconst(float c) { Dual r; r.v = c; for (int i = 0; i < 6; ++i) r.d[i] = 0.f; return r; }
__device__ __forceinline__ Dual dvar(float c, int i) { Dual r = dconst(c); r.d[i] = 1.f; return r; }
__device__ __forceinline__ Dual operator+(Dual a, Dual b) { Dual r; r.v = a.v + b.v; for (int i = 0; i < 6; ++i) r.d[i] = a.d[i] + b.d[i]; return r; }
__device__ __forceinline__ Dual operator-(Dual a, Dual b) { Dual r; r.v = a.v - b.v; for (int i = 0; i < 6; ++i) r.d[i] = a.d[i] - b.d[i]; return r; }
__device__ __forceinline__ Dual operator-(Dual a) { Dual r; r.v = -a.v; for (int i = 0; i < 6; ++i) r.d[i] = -a.d[i]; return r; }
__device__ __forceinline__ Dual operator*(Dual a, Dual b) { Dual r; r.v = a.v * b.v; for (int i = 0; i < 6; ++i) r.d[i] = a.d[i] * b.v + a.v * b.d[i]; return r; }
__device__ __forceinline__ Dual operator*(float a, Dual b) { Dual r; r.v = a * b.v; for (int i = 0; i < 6; ++i) r.d[i] = a * b.d[i]; return r; }
__device__ __forceinline__ Dual operator/(Dual a, Dual b) {
  Dual r; r.v = a.v / b.v;
  for (int i = 0; i < 6; ++i) r.d[i] = (a.d[i] - r.v * b.d[i]) / b.v;
  return r;
}
__device__ __forceinline__ Dual dsqrt(Dual a) { Dual r; r.v = sqrtf(a.v); for (int i = 0; i < 6; ++i) r.d[i] = a.v > 0.f ? a.d[i] / (2.f * r.v) : 0.f; return r; }
__device__ __forceinline__ Dual dsin(Dual a) { Dual r; r.v = sinf(a.v); const float c = cosf(a.v); for (int i = 0; i < 6; ++i) r.d[i] = c * a.d[i]; return r; }
__device__ __forceinline__ Dual dcos(Dual a) { Dual r; r.v = cosf(a.v); const float s = -sinf(a.v); for (int i = 0; i < 6; ++i) r.d[i] = s * a.d[i]; return r; }

// se3.exp on duals (same formulas as se3_math.cuh): g[12] = rows 0..2 of the 4x4 matrix
__device__ void se3_exp_dual(const float* x, Dual* g) {
  Dual w[3], v[3];
  for (int i = 0; i < 3; ++i) { w[i] = dvar(x[i], i); v[i] = dvar(x[3 + i], 3 + i); }
  const Dual t2 = w[0] * w[0] + w[1] * w[1] + w[2] * w[2];
  const Dual t = dsqrt(t2);
  Dual s1, s2, s3;
  const Dual one = dconst(1.f);
  if (fabsf(t.v) < 0.01f) {
    s1 = one - (1.f / 6.f) * t2 * (one - (1.f / 20.f) * t2 * (one - (1.f / 42.f) * t2));
    s2 = 0.5f * (one - (1.f / 12.f) * t2 * (one - (1.f / 30.f) * t2 * (one - (1.f / 56.f) * t2)));
    s3 = (1.f / 6.f) * (one - (1.f / 20.f) * t2 * (one - (1.f / 42.f) * t2 * (one - (1.f / 72.f) * t2)));
  } else {
    const Dual sn = dsin(t), cs = dcos(t);
    s1 = sn / t;
    s2 = (one - cs) / t2;
    s3 = (t - sn) / (t2 * t);
  }
  const Dual z = dconst(0.f);
  const Dual W[9] = {z, -w[2], w[1], w[2], z, -w[0], -w[1], w[0], z};
  Dual S[9];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) S[i * 3 + j] = W[i * 3] * W[j] + W[i * 3 + 1] * W[3 + j] + W[i * 3 + 2] * W[6 + j];
  for (int i = 0; i < 3; ++i) {
    Dual pp = z;
    for (int j = 0; j < 3; ++j) {
      const Dual id = dconst(i == j ? 1.f : 0.f);
      g[i * 4 + j] = id + s1 * W[i * 3 + j] + s2 * S[i * 3 + j];
      pp = pp + (id + s2 * W[i * 3 + j] + s3 * S[i * 3 + j]) * v[j];
    }
    g[i * 4 + 3] = pp;
  }
}

// One CTA per pair.  dpts [B,n,3] = d loss / d (R p + t);  adds J^T (dR, dt) (+ the comp term) to dout6 [B,6].
__global__ void __launch_bounds__(256) pose_grad_kernel(const float* __restrict__ out6, const float* __restrict__ pts,
                                                        const float* __restrict__ dpts, int n,
                                                        const float* __restrict__ igt, float comp_scale, int B,
                                                        float beta, float* __restrict__ dout6) {
  __shared__ float red[9];
  __shared__ float dmat[12];
  const int b = blockIdx.x;
  float acc[12];
  for (int i = 0; i < 12; ++i) acc[i] = 0.f;
  if (dpts) {
    for (int i = threadIdx.x; i < n; i += 256) {
      const float* p = pts + ((size_t)b * n + i) * 3;
      const float* d = dpts + ((size_t)b * n + i) * 3;
      for (int r = 0; r < 3; ++r) {
        acc[r * 4 + 0] = fmaf(d[r], p[0], acc[r * 4 + 0]);
        acc[r * 4 + 1] = fmaf(d[r], p[1], acc[r * 4 + 1]);
        acc[r * 4 + 2] = fmaf(d[r], p[2], acc[r * 4 + 2]);
        acc[r * 4 + 3] += d[r];
      }
    }
  }
  for (int i = 0; i < 12; ++i) {
    const float s = block_sum_256(acc[i], red);
    if (threadIdx.x == 0) dmat[i] = s;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    Dual g[12];
    se3_exp_dual(out6 + b * 6, g);
    if (igt) {
      // comp: L = comp_scale * sum_{b,r,c} (A - I)^2 / B, A = g igt;  dL/dg[r,k] = sum_c 2 (A-I)[r,c] igt[k,c] * comp_scale / B
      const float* H = igt + (size_t)b * 16;
      float Gm[16];
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 4; ++c) Gm[r * 4 + c] = g[r * 4 + c].v;
      Gm[12] = 0.f; Gm[13] = 0.f; Gm[14] = 0.f; Gm[15] = 1.f;
      float dA[16];
      for (int r = 0; r < 4; ++r)
        for (int c = 0; c < 4; ++c) {
          float a = 0.f;
          for (int k = 0; k < 4; ++k) a = fmaf(Gm[r * 4 + k], H[k * 4 + c], a);
          dA[r * 4 + c] = 2.f * (a - (r == c ? 1.f : 0.f)) * comp_scale / (float)B;
        }
      for (int r = 0; r < 3; ++r)
        for (int k = 0; k < 4; ++k) {
          float s = 0.f;
          for (int c = 0; c < 4; ++c) s = fmaf(dA[r * 4 + c], H[k * 4 + c], s);
          dmat[r * 4 + k] += s;
        }
    }
    for (int i = 0; i < 6; ++i) {
      float s = 0.f;
      for (int e = 0; e < 12; ++e) s = fmaf(dmat[e], g[e].d[i], s);
      dout6[b * 6 + i] = (beta != 0.f ? beta * dout6[b * 6 + i] : 0.f) + s;
    }
  }
}

// se3.exp backward on its own (autograd of se3.exp): dtwist[b,:] = sum_e dg[b,e] dg_e/dtwist over the 12 entries of
// rows 0..2 of g [B,4,4] (row 3 is constant).  One thread per item.
__global__ void __launch_bounds__(128) se3_exp_bwd_kernel(const float* __restrict__ twist, const float* __restrict__ dg,
                                                          int B, float* __restrict__ dtwist) {
  const int b = blockIdx.x * 128 + threadIdx.x;
  if (b >= B) return;
  Dual g[12];
  se3_exp_dual(twist + (size_t)b * 6, g);
  const float* d = dg + (size_t)b * 16;
  for (int i = 0; i < 6; ++i) {
    float s = 0.f;
    for (int e = 0; e < 12; ++e) s = fmaf(d[e], g[e].d[i], s);
    dtwist[(size_t)b * 6 + i] = s;
  }
}

// comp backward (the comp term of pose_grad_kernel on a [B,4,4] g): L = sum_{b,r,c} (A - I)^2 / B with A = g igt,
// dg[b,r,k] = dloss * 2/B * sum_c (A - I)[r,c] igt[b,k,c].  One thread per entry of dg.
__global__ void __launch_bounds__(256) comp_bwd_kernel(const float* __restrict__ g, const float* __restrict__ igt, int B,
                                                       const float* __restrict__ dloss, float* __restrict__ dg) {
  const long long e = (long long)blockIdx.x * 256 + threadIdx.x;
  if (e >= 16LL * B) return;
  const long long b = e >> 4;
  const int r = (int)(e >> 2) & 3, k = (int)e & 3;
  const float* G = g + b * 16 + r * 4;
  const float* H = igt + b * 16;
  float s = 0.f;
  for (int c = 0; c < 4; ++c) {
    float a = G[0] * H[c];
    a = fmaf(G[1], H[4 + c], a);
    a = fmaf(G[2], H[8 + c], a);
    a = fmaf(G[3], H[12 + c], a);
    s = fmaf(a - (r == c ? 1.f : 0.f), H[k * 4 + c], s);
  }
  dg[e] = 2.f * dloss[0] / (float)B * s;
}

// =============================================================================== Adam (torch.optim.Adam semantics)
__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                   float* __restrict__ v, long long n, float lr, float b1, float b2,
                                                   float eps, float bc1, float bc2_sqrt, float grad_scale) {
  const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const float gi = g[i] * grad_scale;
  const float mi = b1 * m[i] + (1.f - b1) * gi;
  const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
  m[i] = mi;
  v[i] = vi;
  const float denom = sqrtf(vi) / bc2_sqrt + eps;
  p[i] -= (lr / bc1) * (mi / denom);
}

}  // namespace
}  // namespace pz

using namespace pz;

extern "C" int pz_sgemm(int transA, int transB, int M, int N, int K, float alpha, const float* A, long long lda,
                        const float* B, long long ldb, float beta, float* C, long long ldc, int batch,
                        long long strideA, long long strideB, long long strideC, int splitk, const float* bias_or_null,
                        int relu, const float* mask_or_null, long long ldmask, const float* residual_or_null,
                        long long ldres, pz_stream_t stream) {
  PZ_REQUIRE(M >= 0 && N >= 0 && K >= 0 && batch >= 0, PZ_ERR_ARG, "pz_sgemm: negative size");
  if (M == 0 || N == 0 || batch == 0) return PZ_OK;
  PZ_REQUIRE(A && B && C, PZ_ERR_ARG, "pz_sgemm: null pointer");
  PZ_REQUIRE(K >= 1, PZ_ERR_ARG, "pz_sgemm: K must be >= 1");
  PZ_REQUIRE(splitk >= 1, PZ_ERR_ARG, "pz_sgemm: splitk must be >= 1");
  PZ_REQUIRE(!(splitk > 1 && (batch > 1 || bias_or_null || relu || mask_or_null || residual_or_null || beta != 0.f)),
             PZ_ERR_UNSUPPORTED, "pz_sgemm: split-K excludes batching and epilogues (C must be pre-zeroed)");
  SgemmArgs p;
  p.A = A; p.B = B; p.C = C;
  // op(A) is M x K: not transposed -> A[m*lda + k]; transposed -> stored K x M: A[k*lda + m]
  p.sam = transA ? 1 : lda; p.sak = transA ? lda : 1;
  p.sbk = transB ? 1 : ldb; p.sbn = transB ? ldb : 1;
  p.ldc = ldc; p.bsa = strideA; p.bsb = strideB; p.bsc = strideC;
  p.M = M; p.N = N; p.K = K; p.splitk = splitk; p.alpha = alpha; p.beta = beta;
  p.bias = bias_or_null; p.relu = relu; p.mask = mask_or_null; p.ldmask = ldmask; p.bsmask = strideC;
  p.residual = residual_or_null; p.ldres = ldres; p.bsres = strideC;
  const int gt = (M <= 64 || N <= 64) ? 64 : 128;          // narrow outputs: 64 x 64 tiles
  const int nz = splitk > 1 ? splitk : batch;
  PZ_REQUIRE((M + gt - 1) / gt <= 65535 && nz <= 65535, PZ_ERR_UNSUPPORTED, "pz_sgemm: grid too large (M=%d batch=%d)", M, batch);
  if (gt == 64) sgemm_dispatch<64>(p, transA, transB, nz, as_stream(stream));
  else sgemm_dispatch<128>(p, transA, transB, nz, as_stream(stream));
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_colsum(const float* x, long long ld, long long M, int N, float beta, float* out, pz_stream_t stream) {
  PZ_REQUIRE(N >= 0 && M >= 0, PZ_ERR_ARG, "pz_colsum: negative size");
  if (N == 0) return PZ_OK;
  PZ_REQUIRE(x && out, PZ_ERR_ARG, "pz_colsum: null pointer");
  // out = beta*out, then partial sums are atomically added (row chunks sized so the grid is a few waves of 148 SMs)
  scale_kernel<<<(N + 255) / 256, 256, 0, as_stream(stream)>>>(out, N, beta);
  PZ_LAUNCH_CHECK();
  if (M == 0) return PZ_OK;
  const int col_ctas = (N + 31) / 32;
  long long chunks = (4LL * kNumSMs + col_ctas - 1) / col_ctas;
  long long rows_per_cta = (M + chunks - 1) / chunks;
  if (rows_per_cta < 64) rows_per_cta = 64;
  chunks = (M + rows_per_cta - 1) / rows_per_cta;
  colsum_kernel<<<dim3(col_ctas, (unsigned)chunks), 256, 0, as_stream(stream)>>>(x, ld, M, N, rows_per_cta, out);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_axpby(long long rows, int cols, float a, const float* x, long long ldx, float b,
                        const float* y_or_null, long long ldy, float* out, long long ldo, pz_stream_t stream) {
  PZ_REQUIRE(rows >= 0 && cols >= 0, PZ_ERR_ARG, "pz_axpby: negative size");
  if (rows == 0 || cols == 0) return PZ_OK;
  PZ_REQUIRE(x && out, PZ_ERR_ARG, "pz_axpby: null pointer");
  const long long n = rows * cols;
  if (ldx == cols && ldo == cols && (!y_or_null || ldy == cols))
    axpby_kernel<<<(unsigned)((n + 255) / 256), 256, 0, as_stream(stream)>>>(n, a, x, b, y_or_null, out);
  else
    axpby2d_kernel<<<(unsigned)((n + 255) / 256), 256, 0, as_stream(stream)>>>(rows, cols, a, x, ldx, b, y_or_null, ldy,
                                                                               out, ldo);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_bias_act(long long rows, int cols, float* x, long long ld, const float* bias_or_null, int relu,
                           pz_stream_t stream) {
  PZ_REQUIRE(rows >= 0 && cols >= 0, PZ_ERR_ARG, "pz_bias_act: negative size");
  if (rows == 0 || cols == 0) return PZ_OK;
  PZ_REQUIRE(x, PZ_ERR_ARG, "pz_bias_act: null pointer");
  bias_act_kernel<<<(unsigned)((rows * cols + 255) / 256), 256, 0, as_stream(stream)>>>(rows, cols, x, ld, bias_or_null, relu);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_relu_gate(long long rows, int cols, const float* dy, long long ldy, const float* mask, long long ldm,
                            float* out, long long ldo, pz_stream_t stream) {
  PZ_REQUIRE(rows >= 0 && cols >= 0, PZ_ERR_ARG, "pz_relu_gate: negative size");
  if (rows == 0 || cols == 0) return PZ_OK;
  PZ_REQUIRE(dy && mask && out, PZ_ERR_ARG, "pz_relu_gate: null pointer");
  relu_gate_kernel<<<(unsigned)((rows * cols + 255) / 256), 256, 0, as_stream(stream)>>>(rows, cols, dy, ldy, mask, ldm,
                                                                                         out, ldo);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_broadcast_rows(const float* src, long long G, int reps, int C, float* dst, long long ldd,
                                 pz_stream_t stream) {
  PZ_REQUIRE(G >= 0 && reps >= 1 && C >= 1, PZ_ERR_ARG, "pz_broadcast_rows: bad size");
  if (G == 0) return PZ_OK;
  PZ_REQUIRE(src && dst, PZ_ERR_ARG, "pz_broadcast_rows: null pointer");
  broadcast_rows_kernel<<<(unsigned)((G * reps * C + 255) / 256), 256, 0, as_stream(stream)>>>(src, G, reps, C, dst, ldd);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_group_sum(const float* x, long long ld, long long G, int K, int C, float* y, pz_stream_t stream) {
  PZ_REQUIRE(G >= 0 && K >= 1 && C >= 1, PZ_ERR_ARG, "pz_group_sum: bad size");
  if (G == 0) return PZ_OK;
  PZ_REQUIRE(x && y, PZ_ERR_ARG, "pz_group_sum: null pointer");
  PZ_REQUIRE(G <= 65535, PZ_ERR_UNSUPPORTED, "pz_group_sum: G > 65535");
  group_sum_kernel<<<dim3((C + 31) / 32, (unsigned)G), 256, 0, as_stream(stream)>>>(x, ld, G, K, C, y);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_bn_point_train_forward(const float* x, int B, int P, int C, const float* gamma, const float* beta,
                                         float* running_mean_or_null, float* running_var_or_null, float momentum,
                                         float eps, int relu, float* y, float* save_mean, float* save_invstd,
                                         pz_stream_t stream) {
  PZ_REQUIRE(x && gamma && beta && y && save_mean && save_invstd, PZ_ERR_ARG, "pz_bn_point_train_forward: null pointer");
  PZ_REQUIRE(B >= 1 && P >= 1 && C >= 1, PZ_ERR_ARG, "pz_bn_point_train_forward: bad size");
  PZ_REQUIRE((running_mean_or_null == nullptr) == (running_var_or_null == nullptr), PZ_ERR_ARG,
             "pz_bn_point_train_forward: running_mean and running_var go together");
  bn_point_fwd_kernel<<<P, 256, 0, as_stream(stream)>>>(x, B, P, C, gamma, beta, running_mean_or_null,
                                                        running_var_or_null, momentum, eps, relu, y, save_mean,
                                                        save_invstd);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_bn_point_train_backward(const float* x, const float* y, const float* dy, int B, int P, int C,
                                          const float* gamma, const float* save_mean, const float* save_invstd,
                                          int relu, int accumulate, float* dx, float* dgamma, float* dbeta,
                                          pz_stream_t stream) {
  PZ_REQUIRE(x && y && dy && gamma && save_mean && save_invstd && dx && dgamma && dbeta, PZ_ERR_ARG,
             "pz_bn_point_train_backward: null pointer");
  PZ_REQUIRE(B >= 1 && P >= 1 && C >= 1, PZ_ERR_ARG, "pz_bn_point_train_backward: bad size");
  bn_point_bwd_kernel<<<P, 256, 0, as_stream(stream)>>>(x, y, dy, B, P, C, gamma, save_mean, save_invstd, relu,
                                                        accumulate, dx, dgamma, dbeta);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_maxpool_forward(const float* x, long long G, int K, int C, float* y, int32_t* arg,
                                  pz_stream_t stream) {
  PZ_REQUIRE(G >= 0 && K >= 1 && C >= 1, PZ_ERR_ARG, "pz_maxpool_forward: bad size");
  if (G == 0) return PZ_OK;
  PZ_REQUIRE(x && y && arg, PZ_ERR_ARG, "pz_maxpool_forward: null pointer");
  PZ_REQUIRE(G <= 2147483647LL, PZ_ERR_UNSUPPORTED, "pz_maxpool_forward: too many groups");
  const bool vec = C % 4 == 0 && ((uintptr_t)x & 15) == 0;
  int threads = ((vec ? C / 4 : C) + 31) / 32 * 32;
  if (threads > 256) threads = 256;
  if (vec) maxpool_fwd_kernel<4><<<(unsigned)G, threads, 0, as_stream(stream)>>>(x, K, C, y, arg);
  else maxpool_fwd_kernel<1><<<(unsigned)G, threads, 0, as_stream(stream)>>>(x, K, C, y, arg);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_maxpool_backward(const float* dy, const float* y, const int32_t* arg, long long G, int K, int C,
                                   int relu_gate, float* dx, pz_stream_t stream) {
  PZ_REQUIRE(G >= 0 && K >= 1 && C >= 1, PZ_ERR_ARG, "pz_maxpool_backward: bad size");
  if (G == 0) return PZ_OK;
  PZ_REQUIRE(dy && y && arg && dx, PZ_ERR_ARG, "pz_maxpool_backward: null pointer");
  PZ_REQUIRE(G <= 2147483647LL, PZ_ERR_UNSUPPORTED, "pz_maxpool_backward: too many groups");
  const bool vec = C % 4 == 0 && C / 4 <= 256 && 256 % (C / 4) == 0 && ((uintptr_t)dy & 15) == 0 && ((uintptr_t)y & 15) == 0 &&
                   ((uintptr_t)arg & 15) == 0 && ((uintptr_t)dx & 15) == 0;
  if (vec) maxpool_bwd_kernel<4><<<(unsigned)G, 256, 0, as_stream(stream)>>>(dy, y, arg, K, C, relu_gate, dx);
  else maxpool_bwd_kernel<1><<<(unsigned)G, 256, 0, as_stream(stream)>>>(dy, y, arg, K, C, relu_gate, dx);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_scatter_add_rows(const float* src, long long ld, int c0, int C, const int64_t* idx, long long M,
                                   long long per_cloud, int N, float* dst, long long ldd, pz_stream_t stream) {
  PZ_REQUIRE(M >= 0 && C >= 0, PZ_ERR_ARG, "pz_scatter_add_rows: negative size");
  if (M == 0 || C == 0) return PZ_OK;
  PZ_REQUIRE(src && idx && dst && per_cloud >= 1 && N >= 1, PZ_ERR_ARG, "pz_scatter_add_rows: bad argument");
  const long long want = (M + 7) / 8;
  const unsigned blocks = (unsigned)(want < 32LL * kNumSMs ? want : 32LL * kNumSMs);
  scatter_add_rows_kernel<<<blocks, 256, 0, as_stream(stream)>>>(src, ld, c0, C, idx, M, per_cloud, N, dst, ldd);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_gather_sub_relu(const float* P, const float* Q, const int64_t* idx, long long groups, int K, int S, int N,
                                  int C, float* out, pz_stream_t stream) {
  PZ_REQUIRE(groups >= 0 && K >= 1 && S >= 1 && N >= 1, PZ_ERR_ARG, "pz_gather_sub_relu: bad size");
  if (groups == 0) return PZ_OK;
  PZ_REQUIRE(P && Q && idx && out, PZ_ERR_ARG, "pz_gather_sub_relu: null pointer");
  PZ_REQUIRE(C >= 4 && C % 4 == 0 && ((uintptr_t)P & 15) == 0 && ((uintptr_t)Q & 15) == 0 && ((uintptr_t)out & 15) == 0,
             PZ_ERR_UNSUPPORTED, "pz_gather_sub_relu: C must be a multiple of 4 and the tensors 16-byte aligned");
  const long long rows = groups * K, want = (rows + 7) / 8;
  const unsigned blocks = (unsigned)(want < 64LL * kNumSMs ? want : 64LL * kNumSMs);
  gather_sub_relu_kernel<<<blocks, 256, 0, as_stream(stream)>>>(P, Q, idx, rows, K, S, N, C, out);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_group_scatter_grad(const float* d, const int64_t* idx, long long groups, int K, int S, int N, int C,
                                     float* dP, float* dQ, pz_stream_t stream) {
  PZ_REQUIRE(groups >= 0 && K >= 1 && S >= 1 && N >= 1, PZ_ERR_ARG, "pz_group_scatter_grad: bad size");
  if (groups == 0) return PZ_OK;
  PZ_REQUIRE(d && idx && dP && dQ, PZ_ERR_ARG, "pz_group_scatter_grad: null pointer");
  PZ_REQUIRE(C >= 4 && C % 4 == 0 && ((uintptr_t)d & 15) == 0 && ((uintptr_t)dQ & 15) == 0, PZ_ERR_UNSUPPORTED,
             "pz_group_scatter_grad: C must be a multiple of 4 and the tensors 16-byte aligned");
  const long long want = (groups + 7) / 8;
  const unsigned blocks = (unsigned)(want < 64LL * kNumSMs ? want : 64LL * kNumSMs);
  group_scatter_grad_kernel<<<blocks, 256, 0, as_stream(stream)>>>(d, idx, groups, K, S, N, C, dP, dQ);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_softmax_forward(const float* S, long long rows, int L, float scale, float* A, pz_stream_t stream) {
  PZ_REQUIRE(rows >= 0 && L >= 1, PZ_ERR_ARG, "pz_softmax_forward: bad size");
  if (rows == 0) return PZ_OK;
  PZ_REQUIRE(S && A, PZ_ERR_ARG, "pz_softmax_forward: null pointer");
  softmax_fwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, as_stream(stream)>>>(S, rows, L, scale, A);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_softmax_backward(const float* A, const float* dA, long long rows, int L, float scale, float* dS,
                                   pz_stream_t stream) {
  PZ_REQUIRE(rows >= 0 && L >= 1, PZ_ERR_ARG, "pz_softmax_backward: bad size");
  if (rows == 0) return PZ_OK;
  PZ_REQUIRE(A && dA && dS, PZ_ERR_ARG, "pz_softmax_backward: null pointer");
  softmax_bwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, as_stream(stream)>>>(A, dA, rows, L, scale, dS);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_cross_entropy(const float* logits, const float* target, int B, int N, int point_major,
                                float grad_scale, float* loss, float* dlogits_or_null, pz_stream_t stream) {
  PZ_REQUIRE(logits && target && loss, PZ_ERR_ARG, "pz_cross_entropy: null pointer");
  PZ_REQUIRE(B >= 1 && N >= 1, PZ_ERR_ARG, "pz_cross_entropy: bad size (mean over an empty set)");
  const long long n = (long long)B * N;
  const long long sb = 2LL * N, sc = point_major ? 1 : N, sn = point_major ? 2 : 1;
  cross_entropy_kernel<<<(unsigned)((n + 255) / 256), 256, 0, as_stream(stream)>>>(logits, target, B, N, sb, sc, sn,
                                                                                   grad_scale, loss, dlogits_or_null);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_pose_grad(const float* out6, const float* pts_or_null, const float* dpts_or_null, int n,
                            const float* igt_or_null, float comp_scale, int B, float beta, float* dout6,
                            pz_stream_t stream) {
  PZ_REQUIRE(B >= 0, PZ_ERR_ARG, "pz_pose_grad: B < 0");
  if (B == 0) return PZ_OK;
  PZ_REQUIRE(out6 && dout6, PZ_ERR_ARG, "pz_pose_grad: null pointer");
  PZ_REQUIRE((pts_or_null == nullptr) == (dpts_or_null == nullptr), PZ_ERR_ARG, "pz_pose_grad: pts and dpts go together");
  pose_grad_kernel<<<B, 256, 0, as_stream(stream)>>>(out6, pts_or_null, dpts_or_null, n, igt_or_null, comp_scale, B, beta,
                                                     dout6);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_se3_exp_backward(const float* twist, const float* dg, int B, float* dtwist, pz_stream_t stream) {
  PZ_REQUIRE(twist && dg && dtwist, PZ_ERR_ARG, "pz_se3_exp_backward: null pointer");
  PZ_REQUIRE(B >= 1, PZ_ERR_ARG, "pz_se3_exp_backward: B must be >= 1");
  se3_exp_bwd_kernel<<<(unsigned)((B + 127) / 128), 128, 0, as_stream(stream)>>>(twist, dg, B, dtwist);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_comp_backward(const float* g, const float* igt, int B, const float* dloss, float* dg,
                                pz_stream_t stream) {
  PZ_REQUIRE(g && igt && dloss && dg, PZ_ERR_ARG, "pz_comp_backward: null pointer");
  PZ_REQUIRE(B >= 1, PZ_ERR_ARG, "pz_comp_backward: B must be >= 1");
  comp_bwd_kernel<<<(unsigned)((16LL * B + 255) / 256), 256, 0, as_stream(stream)>>>(g, igt, B, dloss, dg);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}

extern "C" int pz_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                            float beta1, float beta2, float eps, int step, float grad_scale, pz_stream_t stream) {
  PZ_REQUIRE(n >= 0 && step >= 1, PZ_ERR_ARG, "pz_adam_step: bad size / step");
  if (n == 0) return PZ_OK;
  PZ_REQUIRE(params && grads && exp_avg && exp_avg_sq, PZ_ERR_ARG, "pz_adam_step: null pointer");
  const float bc1 = 1.f - powf(beta1, (float)step);
  const float bc2 = 1.f - powf(beta2, (float)step);
  adam_kernel<<<(unsigned)((n + 255) / 256), 256, 0, as_stream(stream)>>>(params, grads, exp_avg, exp_avg_sq, n, lr, beta1,
                                                                          beta2, eps, bc1, sqrtf(bc2), grad_scale);
  PZ_LAUNCH_CHECK();
  return PZ_OK;
}
