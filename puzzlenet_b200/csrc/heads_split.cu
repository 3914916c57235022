// Boundary heads (model5_b.py:738-754) at fp32 tolerance on the tensor cores: two chained-MMA kernels
// (mma.sync m16n8k16, fp16 x fp16 -> fp32) in which every activation and every weight is a hi / lo fp16 pair and every
// product is hi*hi + hi*lo + lo*hi.  The accumulator fragments of one layer, split again, ARE the A fragments of the
// next, so activations never leave registers between layers.  One warp = 32 points; x_feature (fp32) is read straight
// into fragments and the local features / logits are written straight from fragments (every warp-wide access covers
// whole 32-byte sectors), so there is no shared-memory staging of activations at all.
// Used by the split path and by the bf16 path (whose x_feature is fp32-accurate already): the logits of both agree with
// the reference to ~1e-6, at 3x the MMA count of the former bf16 chains -- the kernels are latency-bound, not MMA-bound.
#include <cuda_fp16.h>

#include "pz_common.cuh"

namespace pz {

namespace {

constexpr int NPTS_H = 1024;
constexpr int HS_WS = 72;                                    // padded fp16 row stride: conflict-free fragment loads
constexpr int PRE_ROWS = 3 * 64, SEG_ROWS = 64 + 32;         // weight rows per plane: pre.w0|w1|w2 ; seg.w0[:, 64:] | seg.w1

__device__ __forceinline__ void mma_f16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
               "{%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  uint32_t h;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h) : "f"(b), "f"(a));
  const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&h));
  uint32_t l;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(l) : "f"(b - hf.y), "f"(a - hf.x));
  hi = h;
  lo = l;
}
struct Frags {
  uint32_t hi[2][4][4], lo[2][4][4];   // [m-tile of 16 points][k-tile of 16 channels][a0..a3]
};
// 32 points x 64 channels of an fp32 [P, 64] tensor -> split A fragments
__device__ __forceinline__ void load_frags(const float* __restrict__ src, int g, int q, Frags& a) {
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int kt = 0; kt < 4; ++kt) {
      const float* t0 = src + (size_t)(mt * 16 + g) * 64 + kt * 16 + q * 2;
      const float2 v0 = *reinterpret_cast<const float2*>(t0), v1 = *reinterpret_cast<const float2*>(t0 + 8 * 64);
      const float2 v2 = *reinterpret_cast<const float2*>(t0 + 8), v3 = *reinterpret_cast<const float2*>(t0 + 8 * 64 + 8);
      split2(v0.x, v0.y, a.hi[mt][kt][0], a.lo[mt][kt][0]);
      split2(v1.x, v1.y, a.hi[mt][kt][1], a.lo[mt][kt][1]);
      split2(v2.x, v2.y, a.hi[mt][kt][2], a.lo[mt][kt][2]);
      split2(v3.x, v3.y, a.hi[mt][kt][3], a.lo[mt][kt][3]);
    }
}
// acc[mt][nt] += A[mt] . W^T for NT n-tiles of a [NT*8, 64] weight block (planes wh / wl in smem, row stride HS_WS)
template <int NT>
__device__ __forceinline__ void layer(const Frags& a, const __half* wh, const __half* wl, int g, int q, float (&acc)[2][NT][4]) {
#pragma unroll
  for (int nt = 0; nt < NT; ++nt)
#pragma unroll
    for (int kt = 0; kt < 4; ++kt) {
      const int off = (nt * 8 + g) * HS_WS + kt * 16 + q * 2;
      const uint32_t h0 = *reinterpret_cast<const uint32_t*>(wh + off), h1 = *reinterpret_cast<const uint32_t*>(wh + off + 8);
      const uint32_t l0 = *reinterpret_cast<const uint32_t*>(wl + off), l1 = *reinterpret_cast<const uint32_t*>(wl + off + 8);
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
        mma_f16(acc[mt][nt], a.lo[mt][kt], h0, h1);
        mma_f16(acc[mt][nt], a.hi[mt][kt], l0, l1);
        mma_f16(acc[mt][nt], a.hi[mt][kt], h0, h1);
      }
    }
}
// act(acc + bias) of a 64-wide layer, split again -> the next layer's A fragments
__device__ __forceinline__ void next_frags(const float (&acc)[2][8][4], const float* bias, int q, bool relu, Frags& a) {
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const float bA = bias[nt * 8 + q * 2], bB = bias[nt * 8 + q * 2 + 1];
      float v0 = acc[mt][nt][0] + bA, v1 = acc[mt][nt][1] + bB, v2 = acc[mt][nt][2] + bA, v3 = acc[mt][nt][3] + bB;
      if (relu) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); v2 = fmaxf(v2, 0.f); v3 = fmaxf(v3, 0.f); }
      split2(v0, v1, a.hi[mt][nt >> 1][(nt & 1) * 2], a.lo[mt][nt >> 1][(nt & 1) * 2]);           // row g
      split2(v2, v3, a.hi[mt][nt >> 1][(nt & 1) * 2 + 1], a.lo[mt][nt >> 1][(nt & 1) * 2 + 1]);   // row g + 8
    }
}
template <int NT>
__device__ __forceinline__ void zero(float (&acc)[2][NT][4]) {
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[mt][nt][i] = 0.f;
}

// fp32 weights -> the fp16 plane images of both sets: per set [pre hi 192 rows][pre lo 192][seg hi 96][seg lo 96], rows of
// HS_WS halves (64 used)
__global__ void __launch_bounds__(256) head_images_kernel(HeadMlp3 pre_a, HeadMlp3 pre_b, HeadMlp3 seg_a, HeadMlp3 seg_b,
                                                          __half* __restrict__ img) {
  const int set = blockIdx.y;
  const HeadMlp3& pre = set == 0 ? pre_a : pre_b;
  const HeadMlp3& seg = set == 0 ? seg_a : seg_b;
  __half* dst = img + (size_t)set * HEAD_SPLIT_IMG_SET;
  for (int e = blockIdx.x * 256 + threadIdx.x; e < (PRE_ROWS + SEG_ROWS) * 64; e += gridDim.x * 256) {
    const int r = e >> 6, c = e & 63;
    float v;
    __half *ph, *pl;
    if (r < PRE_ROWS) {
      const float* w = r < 64 ? pre.w0 : (r < 128 ? pre.w1 : pre.w2);
      v = w[(r & 63) * 64 + c];
      ph = dst + (size_t)r * HS_WS + c;
      pl = ph + (size_t)PRE_ROWS * HS_WS;
    } else {
      const int rr = r - PRE_ROWS;
      v = rr < 64 ? seg.w0[rr * 128 + 64 + c] : seg.w1[(rr - 64) * 64 + c];   // local half of layer 0: columns 64..127
      ph = dst + (size_t)(2 * PRE_ROWS + rr) * HS_WS + c;
      pl = ph + (size_t)SEG_ROWS * HS_WS;
    }
    const __half hi = __float2half_rn(v);
    *ph = hi;
    *pl = __float2half_rn(v - __half2float(hi));
  }
}

// MLPLocalPre{Fpc,Rpc} (model5_b.py:738-739): three 64 -> 64 layers (ReLU after the first two); writes the local
// features (fp32 [P,64]) and, per 128-point tile, their column maxima (tilemax [cloud][8][64]) for the global max-pool
// of model5_b.py:741-744
__global__ void __launch_bounds__(128) head_pre_split_kernel(const float* __restrict__ xfeat, HeadMlp3 wa, HeadMlp3 wb,
                                                             const __half* __restrict__ img, int B, int reps,
                                                             float* __restrict__ local, float* __restrict__ tilemax) {
  extern __shared__ __align__(16) uint8_t hp_smem[];
  __half* ws = reinterpret_cast<__half*>(hp_smem);                         // [2 planes][192 rows][HS_WS]
  float* bs = reinterpret_cast<float*>(ws + 2 * PRE_ROWS * HS_WS);         // [3][64]
  float* cmax = bs + 3 * 64;                                               // [4][64]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, q = lane & 3;
  const int cloud = (int)(((size_t)blockIdx.x * reps * 128) / NPTS_H);
  const int set = cloud / B;
  const HeadMlp3& w = set == 0 ? wa : wb;
  pdl_enter();   // the images may be the direct predecessor's (head_images_kernel)
  {
    const uint4* src = reinterpret_cast<const uint4*>(img + (size_t)set * HEAD_SPLIT_IMG_SET);
    uint4* dst = reinterpret_cast<uint4*>(ws);
    for (int i = tid; i < 2 * PRE_ROWS * HS_WS / 8; i += 128) dst[i] = src[i];
  }
  if (tid < 64) {
    bs[tid] = w.b0[tid];
    bs[64 + tid] = w.b1[tid];
    bs[128 + tid] = w.b2[tid];
  }
  __syncthreads();
  const __half* wl = ws + PRE_ROWS * HS_WS;
#pragma unroll 1
  for (int rep = 0; rep < reps; ++rep) {
    const int tile_id = blockIdx.x * reps + rep;
    const size_t p0 = (size_t)tile_id * 128 + warp * 32;
    Frags a;
    load_frags(xfeat + p0 * 64, g, q, a);
    float acc[2][8][4];
#pragma unroll 1
    for (int l = 0; l < 2; ++l) {
      zero<8>(acc);
      layer<8>(a, ws + l * 64 * HS_WS, wl + l * 64 * HS_WS, g, q, acc);
      next_frags(acc, bs + l * 64, q, true, a);
    }
    zero<8>(acc);
    layer<8>(a, ws + 2 * 64 * HS_WS, wl + 2 * 64 * HS_WS, g, q, acc);
    // local features (no ReLU): fp32 stores straight from the fragments + column maxima over the warp's 32 points
    float* dst = local + p0 * 64;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const int col = nt * 8 + q * 2;
      const float bA = bs[128 + col], bB = bs[128 + col + 1];
      float mA = -INFINITY, mB = -INFINITY;
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
        const float2 r0 = make_float2(acc[mt][nt][0] + bA, acc[mt][nt][1] + bB);
        const float2 r1 = make_float2(acc[mt][nt][2] + bA, acc[mt][nt][3] + bB);
        *reinterpret_cast<float2*>(dst + (size_t)(mt * 16 + g) * 64 + col) = r0;
        *reinterpret_cast<float2*>(dst + (size_t)(mt * 16 + g + 8) * 64 + col) = r1;
        mA = fmaxf(mA, fmaxf(r0.x, r1.x));
        mB = fmaxf(mB, fmaxf(r0.y, r1.y));
      }
#pragma unroll
      for (int o = 4; o < 32; o <<= 1) {   // over the 8 row groups g
        mA = fmaxf(mA, __shfl_xor_sync(0xffffffffu, mA, o));
        mB = fmaxf(mB, __shfl_xor_sync(0xffffffffu, mB, o));
      }
      if (g == 0) {
        cmax[warp * 64 + col] = mA;
        cmax[warp * 64 + col + 1] = mB;
      }
    }
    __syncthreads();
    if (tid < 64)
      tilemax[((size_t)cloud * 8 + (tile_id & 7)) * 64 + tid] =
          fmaxf(fmaxf(cmax[tid], cmax[64 + tid]), fmaxf(cmax[128 + tid], cmax[192 + tid]));
    __syncthreads();   // cmax is rewritten by the next repetition
  }
}

// MLP{Fpcb,Rpcb} (model5_b.py:745-754): relu(W0 [g ; local] + b0) -> relu(W1 . + b1) -> W2 . + b2, logits as [B,2,1024].
// g = the MRPC cloud's global max for BOTH heads (D6); its half of layer 0 is a per-cloud bias computed in the prologue
// (fp32 FMAs); the last layer (32 -> 2) runs on the fp32 fragments.
// pairs == null: cloud c of the 2B (set = c / B, b = c % B) reads local[c] and the tile maxima of cloud B + b, and writes
// row b of de_a / de_b.  pairs [B,2]: every cloud is a pair of set 0: pair b reads local[pairs[b,0]] and the tile maxima
// of row pairs[b,1], and writes row b of de_a.
__global__ void __launch_bounds__(128) head_seg_split_kernel(const float* __restrict__ local, HeadMlp3 wa, HeadMlp3 wb,
                                                             const __half* __restrict__ img, int B, int reps,
                                                             const float* __restrict__ tilemax, float* __restrict__ de_a,
                                                             float* __restrict__ de_b, const int64_t* __restrict__ pairs) {
  __shared__ __align__(16) __half wseg[2 * SEG_ROWS * HS_WS];   // [hi: W0 local 64 rows, W1 32 rows][lo: same]
  __shared__ float gs[64], gb[64], b1s[32], w2s[64], b2s[2];
  const __half *w0h = wseg, *w1h = wseg + 64 * HS_WS, *w0l = wseg + SEG_ROWS * HS_WS, *w1l = w0l + 64 * HS_WS;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, q = lane & 3;
  const int cloud = (int)(((size_t)blockIdx.x * reps * 128) / NPTS_H), set = cloud / B, b = cloud - set * B;
  const HeadMlp3& w = set == 0 ? wa : wb;
  pdl_enter();
  {
    const uint4* src = reinterpret_cast<const uint4*>(img + (size_t)set * HEAD_SPLIT_IMG_SET + 2 * PRE_ROWS * HS_WS);
    uint4* dst = reinterpret_cast<uint4*>(wseg);
    for (int i = tid; i < 2 * SEG_ROWS * HS_WS / 8; i += 128) dst[i] = src[i];
  }
  const size_t src = pairs ? (size_t)pairs[2 * b] : (size_t)cloud;   // cloud of the local features
  if (tid < 64) {
    const float* tm = tilemax + ((size_t)(pairs ? pairs[2 * b + 1] : B + b) * 8) * 64 + tid;   // the mrpc cloud of pair b
    float m = tm[0];
#pragma unroll
    for (int i = 1; i < 8; ++i) m = fmaxf(m, tm[i * 64]);
    gs[tid] = m;
    w2s[tid] = w.w2[tid];
  }
  if (tid < 32) b1s[tid] = w.b1[tid];
  if (tid < 2) b2s[tid] = w.b2[tid];
  __syncthreads();
  if (tid < 64) {
    float v = w.b0[tid];
    const float* wr = w.w0 + tid * 128;
    for (int i = 0; i < 64; ++i) v = fmaf(wr[i], gs[i], v);
    gb[tid] = v;
  }
  __syncthreads();
#pragma unroll 1
  for (int rep = 0; rep < reps; ++rep) {
    const size_t p0 = ((size_t)blockIdx.x * reps + rep) * 128 + warp * 32;
    const int n0 = (int)(p0 - (size_t)cloud * NPTS_H);
    Frags a;
    load_frags(local + (src * NPTS_H + n0) * 64, g, q, a);
    float acc[2][8][4];
    zero<8>(acc);
    layer<8>(a, w0h, w0l, g, q, acc);
    next_frags(acc, gb, q, true, a);
    float h1[2][4][4];
    zero<4>(h1);
    layer<4>(a, w1h, w1l, g, q, h1);
    // layer 2 (32 -> 2) on the fp32 fragments: this thread holds 8 of the 32 hidden channels of its 4 rows
    float o[4][2];
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j][0] = o[j][1] = 0.f;
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      const int col = nt * 8 + q * 2;
      const float bA = b1s[col], bB = b1s[col + 1];
      const float wA0 = w2s[col], wB0 = w2s[col + 1], wA1 = w2s[32 + col], wB1 = w2s[32 + col + 1];
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          const float hA = fmaxf(h1[mt][nt][2 * hf] + bA, 0.f), hB = fmaxf(h1[mt][nt][2 * hf + 1] + bB, 0.f);
          const int j = 2 * mt + hf;
          o[j][0] = fmaf(wA0, hA, fmaf(wB0, hB, o[j][0]));
          o[j][1] = fmaf(wA1, hA, fmaf(wB1, hB, o[j][1]));
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        o[j][c] += __shfl_xor_sync(0xffffffffu, o[j][c], 1);
        o[j][c] += __shfl_xor_sync(0xffffffffu, o[j][c], 2);
      }
    if (q == 0) {
      float* de = set == 0 ? de_a : de_b;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int n = n0 + g + 8 * j;
        de[((size_t)b * 2 + 0) * NPTS_H + n] = o[j][0] + b2s[0];
        de[((size_t)b * 2 + 1) * NPTS_H + n] = o[j][1] + b2s[1];
      }
    }
  }
}

}  // namespace

// fp16 plane images of both heads' weights (img: 2 * HEAD_SPLIT_IMG_SET halves), skipped when the caller vouches for them
static int build_images(const HeadMlp3& pre_f, const HeadMlp3& pre_r, const HeadMlp3& seg_f, const HeadMlp3& seg_r,
                        bool reuse_images, __half* img, cudaStream_t st) {
  if (!reuse_images) {
    head_images_kernel<<<dim3(8, 2), 256, 0, st>>>(pre_f, pre_r, seg_f, seg_r, img);
    PZ_LAUNCH_CHECK();
  }
  return 0;
}

// boundary heads of predict5 for 2B clouds (clouds [0,B) = fpc -> *_fpc weights and de_fpcb, [B,2B) = mrpc):
// xfeat [2B*1024, 64] fp32 -> de_fpcb / de_mrpcb [B,2,1024].  local [2B*1024, 64] fp32 and tilemax [2B*8*64] receive the
// per-cloud state, img (2 * HEAD_SPLIT_IMG_SET halves) holds the weight images: rebuilt unless reuse_images.
int launch_heads_split(const float* xfeat, const HeadMlp3& pre_f, const HeadMlp3& pre_r, const HeadMlp3& seg_f,
                       const HeadMlp3& seg_r, int B, bool reuse_images, void* img, float* local, float* tilemax,
                       float* de_fpcb, float* de_mrpcb, cudaStream_t st) {
  PZ_REQUIRE(xfeat && img && local && tilemax && de_fpcb && de_mrpcb, PZ_ERR_ARG, "heads_split: null pointer");
  __half* im = static_cast<__half*>(img);
  PZ_TRY(build_images(pre_f, pre_r, seg_f, seg_r, reuse_images, im, st));
  const int P = 2 * B * NPTS_H, reps = 4;
  const size_t pre_smem = (size_t)2 * PRE_ROWS * HS_WS * sizeof(__half) + (3 * 64 + 4 * 64) * sizeof(float);
  PZ_CUDA(cudaFuncSetAttribute(head_pre_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pre_smem));
  PZ_CUDA(launch_pdl(head_pre_split_kernel, dim3(P / (128 * reps)), dim3(128), pre_smem, st, xfeat, pre_f, pre_r, (const __half*)im, B, reps,
                     local, tilemax));
  PZ_LAUNCH_CHECK();
  PZ_CUDA(launch_pdl(head_seg_split_kernel, dim3(P / (128 * reps)), dim3(128), 0, st, (const float*)local, seg_f, seg_r, (const __half*)im, B,
                     reps, (const float*)tilemax, de_fpcb, de_mrpcb, (const int64_t*)nullptr));
  PZ_LAUNCH_CHECK();
  return 0;
}

// the fpc boundary head of n pairs from per-piece state (pz_predict_pairs): pair p reads local_fpc[pairs[p,0]]
// ([P*1024, 64]) and the tile maxima tilemax_mrpc[pairs[p,1]] ([P*8*64]) and writes de_fpcb[p] ([n,2,1024])
int launch_seg_pairs_split(const HeadMlp3& pre_f, const HeadMlp3& pre_r, const HeadMlp3& seg_f, const HeadMlp3& seg_r,
                           bool reuse_images, void* img, const float* local_fpc, const float* tilemax_mrpc,
                           const int64_t* pairs, int n, float* de_fpcb, cudaStream_t st) {
  PZ_REQUIRE(img && local_fpc && tilemax_mrpc && pairs && de_fpcb, PZ_ERR_ARG, "heads_split: null pointer");
  __half* im = static_cast<__half*>(img);
  PZ_TRY(build_images(pre_f, pre_r, seg_f, seg_r, reuse_images, im, st));
  const int reps = 4;   // 8 tiles per pair: every CTA stays inside one pair
  PZ_CUDA(launch_pdl(head_seg_split_kernel, dim3(n * NPTS_H / (128 * reps)), dim3(128), 0, st, local_fpc, seg_f, seg_f,
                     (const __half*)im, n, reps, tilemax_mrpc, de_fpcb, (float*)nullptr, pairs));
  PZ_LAUNCH_CHECK();
  return 0;
}

}  // namespace pz
