// PuzzleNet encoder + pair heads on sm_100a (fp32-faithful path).
// Reference: model5_b.py:443-478 (PCTransformer_nonsort.forward), :92-101 (layerAttention),
// :67-75 (scaled_dot_production), :672-759 (TouchedRegraster.predict5); se_math/se3.py:57-80.
//
// Both encoders of predict5 run as ONE batch of 2B clouds (cloud c uses weight set c / B), so
// every launch covers 128 clouds at B=64 instead of 64 -- FPS, the latency-bound stage, then
// occupies 128 of the 148 SMs.

#include <algorithm>
#include <climits>
#include <functional>

#include <cuda_fp16.h>

#include "pz_common.cuh"
#include "se3_math.cuh"

namespace pz {

constexpr int NPTS = 1024;  // BatchNorm1d(1024) over the point index pins N (SURVEY.md D7)
constexpr int S1 = 512, S2 = 256, KNN = 32;
constexpr int D0 = 64, C1A = 128, C1B = 128, C2A = 256, C2B = 256, LATT = 256, CATT = 256;

// ------------------------------------------------------------------ stem (model5_b.py:447-448)
struct StemW {
  const float *w1, *b1, *w2, *b2;
  const float *g1, *be1, *m1, *v1, *g2, *be2, *m2, *v2;
};

__global__ void __launch_bounds__(128) stem_kernel(const float* __restrict__ xyz, StemW wa, StemW wb,
                                                   int clouds_per_set, float* __restrict__ out) {
  __shared__ __align__(16) float w2s[64 * 64];
  __shared__ float w1s[64 * 3], b1s[64], b2s[64];
  const size_t p = (size_t)blockIdx.x * 128 + threadIdx.x;  // global point id
  const int cloud = (int)(p / NPTS);                        // uniform per block (128 | 1024)
  const int n = (int)(p - (size_t)cloud * NPTS);
  const StemW& w = (cloud / clouds_per_set) == 0 ? wa : wb;
  for (int i = threadIdx.x; i < 64 * 64; i += 128) w2s[i] = w.w2[i];
  for (int i = threadIdx.x; i < 64 * 3; i += 128) w1s[i] = w.w1[i];
  if (threadIdx.x < 64) {
    b1s[threadIdx.x] = w.b1[threadIdx.x];
    b2s[threadIdx.x] = w.b2[threadIdx.x];
  }
  __syncthreads();
  // eval-mode BatchNorm1d over the point index: y = x*alpha_n + beta_n
  const float a1 = w.g1[n] * (1.0f / sqrtf(w.v1[n] + 1e-5f));
  const float c1 = w.be1[n] - w.m1[n] * a1;
  const float a2 = w.g2[n] * (1.0f / sqrtf(w.v2[n] + 1e-5f));
  const float c2 = w.be2[n] - w.m2[n] * a2;
  const float x = xyz[p * 3], y = xyz[p * 3 + 1], z = xyz[p * 3 + 2];
  float h[64];
#pragma unroll
  for (int k = 0; k < 64; ++k) {
    float v = b1s[k];
    v = fmaf(w1s[k * 3 + 0], x, v);
    v = fmaf(w1s[k * 3 + 1], y, v);
    v = fmaf(w1s[k * 3 + 2], z, v);
    h[k] = fmaxf(fmaf(v, a1, c1), 0.f);
  }
  float* o = out + p * 64;
#pragma unroll 1
  for (int k0 = 0; k0 < 64; k0 += 4) {
    float r[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float4* wr = reinterpret_cast<const float4*>(&w2s[(k0 + u) * 64]);
      float v = b2s[k0 + u];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        float4 ww = wr[i];
        v = fmaf(ww.x, h[i * 4 + 0], v);
        v = fmaf(ww.y, h[i * 4 + 1], v);
        v = fmaf(ww.z, h[i * 4 + 2], v);
        v = fmaf(ww.w, h[i * 4 + 3], v);
      }
      r[u] = fmaxf(fmaf(v, a2, c2), 0.f);
    }
    *reinterpret_cast<float4*>(o + k0) = make_float4(r[0], r[1], r[2], r[3]);
  }
}

__device__ __forceinline__ void stem_mma(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
               "{%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void stem_mma_f16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
               "{%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// 128-point tiles per CTA of stem_tc_kernel (the tiles of one CTA belong to one cloud: reps | 8)
constexpr int HD_REPS = 4;
constexpr int STEM_WS = 72;
constexpr size_t STEM_TC_SMEM = 4 * 32 * STEM_WS * sizeof(float) + 64 * sizeof(float4) + 64 * sizeof(float) +
                                2 * 64 * STEM_WS * sizeof(__nv_bfloat16);
// bf16-path stem: layer 1 (3 -> 64) + BN + ReLU is computed straight into mma.sync A fragments, layer 2 (64 -> 64) runs
// on the tensor cores (m16n8k16, bf16 x bf16 -> fp32; 1 GFLOP per forward does not warrant a tcgen05 pipeline) as a split
// product (h = hi + lo, W = hi + lo; hi*hi + hi*lo + lo*hi, error ~2^-17) because x_feature is an output and feeds both
// the grouped MLP and the boundary heads, BN + ReLU on the accumulator fragments, and the [32 points x 64] tile of each warp leaves through shared memory as one
// contiguous 8 KB (fp32) + 4 KB (bf16) block.  The fp32 path keeps stem_kernel (FFMA, 1e-4 parity).
// F16 (split path): the halves are fp16 (11 + 11 mantissa bits: x_feature to ~1e-6), W2's hi | lo image is built from
// the fp32 weights by the CTA itself, and the 16-bit outputs are the fp16 hi / lo PLANES of x_feature (out_b = hi plane,
// out_lo = lo plane) that the split row GEMM of layer 1 consumes.
template <bool F16>
__global__ void __launch_bounds__(128) stem_tc_kernel(const float* __restrict__ xyz, StemW wa, StemW wb,
                                                      const __nv_bfloat16* __restrict__ w2img_a,
                                                      const __nv_bfloat16* __restrict__ w2img_b,
                                                      int clouds_per_set, int reps, float* __restrict__ out,
                                                      __nv_bfloat16* __restrict__ out_b, __half* __restrict__ out_lo) {
  constexpr int WS = STEM_WS;   // padded row strides: conflict-free fragment loads / stores
  extern __shared__ __align__(16) uint8_t stem_smem[];
  float* stage_all = reinterpret_cast<float*>(stem_smem);                               // [4][32 * WS]
  float4* w1p = reinterpret_cast<float4*>(stage_all + 4 * 32 * WS);                     // (w1[c][0..2], b1[c])
  float* b2s = reinterpret_cast<float*>(w1p + 64);
  __nv_bfloat16* w2b = reinterpret_cast<__nv_bfloat16*>(b2s + 64);                      // hi, then lo: [2][64 * WS]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, q = lane & 3;
  const int cloud = (int)(((size_t)blockIdx.x * reps * 128) / NPTS);   // uniform per block (128 reps | 1024)
  const StemW& w = (cloud / clouds_per_set) == 0 ? wa : wb;
  if (F16) {   // W2 hi | lo fp16 images from the fp32 weights ([64 out][64 in] row-major)
    __half* w2h = reinterpret_cast<__half*>(w2b);
    for (int i = tid; i < 64 * 64; i += 128) {
      const float v = w.w2[i];
      const __half hi = __float2half_rn(v);
      w2h[(i >> 6) * WS + (i & 63)] = hi;
      w2h[64 * WS + (i >> 6) * WS + (i & 63)] = __float2half_rn(v - __half2float(hi));
    }
  } else {   // W2 hi | lo images ([2][64, WS] bf16, written by the weight pack): a straight 16-byte copy
    const uint4* src = reinterpret_cast<const uint4*>((cloud / clouds_per_set) == 0 ? w2img_a : w2img_b);
    uint4* dst = reinterpret_cast<uint4*>(w2b);
    for (int i = tid; i < 2 * 64 * WS / 8; i += 128) dst[i] = src[i];
  }
  if (tid < 64) {
    w1p[tid] = make_float4(w.w1[tid * 3], w.w1[tid * 3 + 1], w.w1[tid * 3 + 2], w.b1[tid]);
    b2s[tid] = w.b2[tid];
  }
  pdl_enter();   // the weights above are model parameters / images packed at least two launches ago; xyz is the predecessor's
  __syncthreads();
#pragma unroll 1
  for (int rep = 0; rep < reps; ++rep) {
  const size_t p0 = ((size_t)blockIdx.x * reps + rep) * 128;   // first point of this 128-point tile
  const int n0 = (int)(p0 - (size_t)cloud * NPTS) + warp * 32;
  // this thread's four rows of the warp tile: g, g + 8, g + 16, g + 24
  float x[4], y[4], z[4], a1[4], c1[4], a2[4], c2[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int r = g + 8 * j, n = n0 + r;
    const float* pp = xyz + (p0 + warp * 32 + r) * 3;
    x[j] = pp[0]; y[j] = pp[1]; z[j] = pp[2];
    a1[j] = w.g1[n] * (1.0f / sqrtf(w.v1[n] + 1e-5f));   // eval-mode BatchNorm1d over the point index
    c1[j] = w.be1[n] - w.m1[n] * a1[j];
    a2[j] = w.g2[n] * (1.0f / sqrtf(w.v2[n] + 1e-5f));
    c2[j] = w.be2[n] - w.m2[n] * a2[j];
  }
  // A fragments of h = relu(bn1(W1 xyz + b1)): [2 m-tiles][4 k-tiles][4 regs]
  uint32_t af[2][4][4], al[2][4][4];
#pragma unroll
  for (int kt = 0; kt < 4; ++kt) {
#pragma unroll
    for (int h2 = 0; h2 < 2; ++h2) {
      const int col = kt * 16 + h2 * 8 + q * 2;
      const float4 wA = w1p[col], wB = w1p[col + 1];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float vA = wA.w, vB = wB.w;
        vA = fmaf(wA.x, x[j], vA); vA = fmaf(wA.y, y[j], vA); vA = fmaf(wA.z, z[j], vA);
        vB = fmaf(wB.x, x[j], vB); vB = fmaf(wB.y, y[j], vB); vB = fmaf(wB.z, z[j], vB);
        const float hA = fmaxf(fmaf(vA, a1[j], c1[j]), 0.f), hB = fmaxf(fmaf(vB, a1[j], c1[j]), 0.f);
        if (F16) {
          const __half2 hh = __floats2half2_rn(hA, hB);
          const float2 hf = __half22float2(hh);
          const __half2 hl = __floats2half2_rn(hA - hf.x, hB - hf.y);
          af[j >> 1][kt][(j & 1) + 2 * h2] = *reinterpret_cast<const uint32_t*>(&hh);
          al[j >> 1][kt][(j & 1) + 2 * h2] = *reinterpret_cast<const uint32_t*>(&hl);
        } else {
          const __nv_bfloat162 hh = __floats2bfloat162_rn(hA, hB);
          const float2 hf = __bfloat1622float2(hh);
          const __nv_bfloat162 hl = __floats2bfloat162_rn(hA - hf.x, hB - hf.y);
          af[j >> 1][kt][(j & 1) + 2 * h2] = *reinterpret_cast<const uint32_t*>(&hh);
          al[j >> 1][kt][(j & 1) + 2 * h2] = *reinterpret_cast<const uint32_t*>(&hl);
        }
      }
    }
  }
  float acc[2][8][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[mt][nt][i] = 0.f;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
    for (int kt = 0; kt < 4; ++kt) {
      const __nv_bfloat16* bp = w2b + (nt * 8 + g) * WS + kt * 16 + q * 2;
      const uint32_t b0 = *reinterpret_cast<const uint32_t*>(bp), b1 = *reinterpret_cast<const uint32_t*>(bp + 8);
      const uint32_t l0 = *reinterpret_cast<const uint32_t*>(bp + 64 * WS), l1 = *reinterpret_cast<const uint32_t*>(bp + 64 * WS + 8);
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
        if (F16) {
          stem_mma_f16(acc[mt][nt], al[mt][kt], b0, b1);   // small terms first
          stem_mma_f16(acc[mt][nt], af[mt][kt], l0, l1);
          stem_mma_f16(acc[mt][nt], af[mt][kt], b0, b1);
        } else {
          stem_mma(acc[mt][nt], al[mt][kt], b0, b1);
          stem_mma(acc[mt][nt], af[mt][kt], l0, l1);
          stem_mma(acc[mt][nt], af[mt][kt], b0, b1);
        }
      }
    }
  }
  // epilogue on the fragments: + b2, BN2, ReLU -> the warp's staging tile
  float* st = stage_all + warp * 32 * WS;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    const int col = nt * 8 + q * 2;
    const float bA = b2s[col], bB = b2s[col + 1];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        const int j = 2 * mt + hf;   // row g + 8 j
        float2 o;
        o.x = fmaxf(fmaf(acc[mt][nt][2 * hf] + bA, a2[j], c2[j]), 0.f);
        o.y = fmaxf(fmaf(acc[mt][nt][2 * hf + 1] + bB, a2[j], c2[j]), 0.f);
        *reinterpret_cast<float2*>(st + (g + 8 * j) * WS + col) = o;
      }
    }
  }
  __syncwarp();
  float* ot = out + (p0 + warp * 32) * 64;   // the warp's 32 rows are one contiguous 8 KB block
#pragma unroll
  for (int it = 0; it < 16; ++it) {
    const int idx = it * 32 + lane, row = idx >> 4, c4 = idx & 15;
    *reinterpret_cast<float4*>(ot + idx * 4) = *reinterpret_cast<const float4*>(st + row * WS + c4 * 4);
  }
  if (F16) {
    uint4* oh = reinterpret_cast<uint4*>(reinterpret_cast<__half*>(out_b) + (p0 + warp * 32) * 64);
    uint4* ol = reinterpret_cast<uint4*>(out_lo + (p0 + warp * 32) * 64);
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int idx = it * 32 + lane, row = idx >> 3, c8 = idx & 7;
      const float4 v0 = *reinterpret_cast<const float4*>(st + row * WS + c8 * 8);
      const float4 v1 = *reinterpret_cast<const float4*>(st + row * WS + c8 * 8 + 4);
      const float f[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
      uint32_t hw[4], lw[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const __half2 hh = __floats2half2_rn(f[2 * e], f[2 * e + 1]);
        const float2 hf = __half22float2(hh);
        const __half2 hl = __floats2half2_rn(f[2 * e] - hf.x, f[2 * e + 1] - hf.y);
        hw[e] = *reinterpret_cast<const uint32_t*>(&hh);
        lw[e] = *reinterpret_cast<const uint32_t*>(&hl);
      }
      oh[idx] = make_uint4(hw[0], hw[1], hw[2], hw[3]);
      ol[idx] = make_uint4(lw[0], lw[1], lw[2], lw[3]);
    }
  } else if (out_b) {
    __nv_bfloat16* ob = out_b + (p0 + warp * 32) * 64;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int idx = it * 32 + lane, row = idx >> 3, c8 = idx & 7;
      const float4 v0 = *reinterpret_cast<const float4*>(st + row * WS + c8 * 8);
      const float4 v1 = *reinterpret_cast<const float4*>(st + row * WS + c8 * 8 + 4);
      __nv_bfloat162 h0 = __floats2bfloat162_rn(v0.x, v0.y), h1 = __floats2bfloat162_rn(v0.z, v0.w);
      __nv_bfloat162 h2 = __floats2bfloat162_rn(v1.x, v1.y), h3 = __floats2bfloat162_rn(v1.z, v1.w);
      uint4 pk;
      pk.x = *reinterpret_cast<uint32_t*>(&h0); pk.y = *reinterpret_cast<uint32_t*>(&h1);
      pk.z = *reinterpret_cast<uint32_t*>(&h2); pk.w = *reinterpret_cast<uint32_t*>(&h3);
      *reinterpret_cast<uint4*>(ob + idx * 8) = pk;
    }
  }
  __syncwarp();   // the staging tile is rewritten by the next repetition
  }
}

// ------------------------------------------------- attention core (model5_b.py:67-75, :98-99)
// One CTA per (cloud, 64 query rows): S = q k^T * scale in smem, row softmax, O = A v.
// out = xres ? xres - O : O.   attn_mode: 0 none, 1 store A, 2 A += , 3 A = (A_old + A) * 0.25
constexpr int AT_ROWS = 64;
__global__ void __launch_bounds__(256) attention_kernel(const float* __restrict__ q, int ldq,
                                                        const float* __restrict__ k, int ldk,
                                                        const float* __restrict__ v, int ldv,
                                                        int L, int Dv, float scale,
                                                        const float* __restrict__ xres, int ldx,
                                                        float* __restrict__ out, int ldo,
                                                        float* __restrict__ attn, int attn_mode,
                                                        const __nv_bfloat16* __restrict__ xres_b, int ldxb,
                                                        __nv_bfloat16* __restrict__ out_b, int ldob) {
  extern __shared__ __align__(16) float at_smem[];
  const int lds = L + 4;
  float* Ss = at_smem;                 // [64][L+4]
  float* T0 = Ss + AT_ROWS * lds;      // 64x64 q^T tile, later V chunk [32][128]
  float* T1 = T0 + 64 * 64;            // 64x64 k^T tile
  const int t = threadIdx.x;
  const int cloud = blockIdx.y;
  const int i0 = blockIdx.x * AT_ROWS;
  const size_t row0 = (size_t)cloud * L;

  {  // q^T tile: T0[d][i]
    const int i = t & 63, dq = (t >> 6) * 16;
    const float* src = q + (row0 + i0 + i) * ldq + dq;
#pragma unroll
    for (int u = 0; u < 16; u += 4) {
      float4 x = *reinterpret_cast<const float4*>(src + u);
      T0[(dq + u + 0) * 64 + i] = x.x; T0[(dq + u + 1) * 64 + i] = x.y;
      T0[(dq + u + 2) * 64 + i] = x.z; T0[(dq + u + 3) * 64 + i] = x.w;
    }
  }
  const int tx = t & 15, ty = t >> 4;
  for (int jc = 0; jc < L; jc += 64) {
    __syncthreads();
    {
      const int j = t & 63, dq = (t >> 6) * 16;
      const float* src = k + (row0 + jc + j) * ldk + dq;
#pragma unroll
      for (int u = 0; u < 16; u += 4) {
        float4 x = *reinterpret_cast<const float4*>(src + u);
        T1[(dq + u + 0) * 64 + j] = x.x; T1[(dq + u + 1) * 64 + j] = x.y;
        T1[(dq + u + 2) * 64 + j] = x.z; T1[(dq + u + 3) * 64 + j] = x.w;
      }
    }
    __syncthreads();
    float acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
#pragma unroll 16
    for (int d = 0; d < 64; ++d) {
      float4 a4 = *reinterpret_cast<const float4*>(&T0[d * 64 + ty * 4]);
      float4 b4 = *reinterpret_cast<const float4*>(&T1[d * 64 + tx * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) acc[x][y] = fmaf(a[x], b[y], acc[x][y]);
    }
#pragma unroll
    for (int x = 0; x < 4; ++x)
      *reinterpret_cast<float4*>(&Ss[(ty * 4 + x) * lds + jc + tx * 4]) =
          make_float4(acc[x][0] * scale, acc[x][1] * scale, acc[x][2] * scale, acc[x][3] * scale);
  }
  __syncthreads();
  {  // softmax over each of the 64 rows; warp w owns rows w*8 .. w*8+7
    const int lane = t & 31, w = t >> 5;
    for (int r = w * 8; r < w * 8 + 8; ++r) {
      float* sr = Ss + r * lds;
      float m = -INFINITY;
      for (int c = lane; c < L; c += 32) m = fmaxf(m, sr[c]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
      float sum = 0.f;
      for (int c = lane; c < L; c += 32) {
        float e = expf(sr[c] - m);
        sr[c] = e;
        sum += e;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      const float inv = 1.0f / sum;
      float* ag = attn ? attn + (row0 + i0 + r) * L : nullptr;
      for (int c = lane; c < L; c += 32) {
        float a = sr[c] * inv;
        sr[c] = a;
        if (attn_mode == 1) ag[c] = a;
        else if (attn_mode == 2) ag[c] += a;
        else if (attn_mode == 3) ag[c] = (ag[c] + a) * 0.25f;
      }
    }
  }
  // O = A v: 128 output columns per pass, thread = 8 rows x 4 cols
  const int px = t & 31, py = t >> 5;
  float* Vs = T0;  // [32][128]
  for (int cb = 0; cb < Dv; cb += 128) {
    float acc[8][4];
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
    for (int j0 = 0; j0 < L; j0 += 32) {
      __syncthreads();
      for (int e = t; e < 32 * 32; e += 256) {  // 32 rows x 32 float4
        const int jr = e >> 5, c4 = (e & 31) * 4;
        *reinterpret_cast<float4*>(&Vs[jr * 128 + c4]) =
            *reinterpret_cast<const float4*>(v + (row0 + j0 + jr) * ldv + cb + c4);
      }
      __syncthreads();
#pragma unroll
      for (int jj = 0; jj < 32; jj += 4) {
        float4 a4[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) a4[r] = *reinterpret_cast<const float4*>(&Ss[(py * 8 + r) * lds + j0 + jj]);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          float4 b4 = *reinterpret_cast<const float4*>(&Vs[(jj + u) * 128 + px * 4]);
#pragma unroll
          for (int r = 0; r < 8; ++r) {
            const float a = u == 0 ? a4[r].x : (u == 1 ? a4[r].y : (u == 2 ? a4[r].z : a4[r].w));
            acc[r][0] = fmaf(a, b4.x, acc[r][0]);
            acc[r][1] = fmaf(a, b4.y, acc[r][1]);
            acc[r][2] = fmaf(a, b4.z, acc[r][2]);
            acc[r][3] = fmaf(a, b4.w, acc[r][3]);
          }
        }
      }
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const size_t row = row0 + i0 + py * 8 + r;
      const int col = cb + px * 4;
      float4 o4 = make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]);
      if (xres) {
        float4 x4 = *reinterpret_cast<const float4*>(xres + row * ldx + col);
        o4 = make_float4(x4.x - o4.x, x4.y - o4.y, x4.z - o4.z, x4.w - o4.w);
      }
      if (xres_b) {
        const uint2 xb = *reinterpret_cast<const uint2*>(xres_b + row * ldxb + col);
        const float2 x01 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&xb.x));
        const float2 x23 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&xb.y));
        o4 = make_float4(x01.x - o4.x, x01.y - o4.y, x23.x - o4.z, x23.y - o4.w);
      }
      if (out) *reinterpret_cast<float4*>(out + row * ldo + col) = o4;
      if (out_b) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(o4.x, o4.y), hi = __floats2bfloat162_rn(o4.z, o4.w);
        *reinterpret_cast<uint2*>(out_b + row * ldob + col) =
            make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
      }
    }
  }
}

static int launch_attention(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv,
                            int clouds, int L, int Dk, int Dv, const float* xres, int ldx, float* out,
                            int ldo, float* attn, int attn_mode, cudaStream_t st,
                            const __nv_bfloat16* xres_b = nullptr, int ldxb = 0, __nv_bfloat16* out_b = nullptr,
                            int ldob = 0) {
  PZ_REQUIRE(Dk == 64 && L % 64 == 0 && L >= 64 && L <= 256 && Dv % 128 == 0 && Dv >= 128, PZ_ERR_UNSUPPORTED,
             "attention: need Dk == 64, L in {64,128,192,256}, Dv %% 128 == 0 (got L=%d Dk=%d Dv=%d)", L, Dk, Dv);
  PZ_REQUIRE(clouds <= 65535, PZ_ERR_UNSUPPORTED, "attention: too many clouds");
  PZ_REQUIRE(ldq % 4 == 0 && ldk % 4 == 0 && ldv % 4 == 0 && ldo % 4 == 0 && (!xres || ldx % 4 == 0), PZ_ERR_ARG,
             "attention: leading dimensions must be multiples of 4");
  size_t smem = ((size_t)AT_ROWS * (L + 4) + 2 * 64 * 64) * sizeof(float);
  PZ_CUDA(cudaFuncSetAttribute(attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid(L / AT_ROWS, clouds);
  attention_kernel<<<grid, 256, smem, st>>>(q, ldq, k, ldk, v, ldv, L, Dv, 1.0f / sqrtf((float)Dk), xres, ldx,
                                            out, ldo, attn, attn_mode, xres_b, ldxb, out_b, ldob);
  PZ_LAUNCH_CHECK();
  return 0;
}

// -------------------------------------------------------------------------- small kernels
// out[(r % rmod) * ldo + (r / rmod) * coloff + c] = max over G consecutive rows of in[., c]
__global__ void __launch_bounds__(256) rowblock_max_kernel(const float* __restrict__ in, int ldi, int G, int N,
                                                           int R, int rmod, int coloff, float* __restrict__ out,
                                                           int ldo) {
  pdl_enter();
  const int r = blockIdx.y;
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c >= N || r >= R) return;
  const float* p = in + (size_t)r * G * ldi + c;
  float m = -INFINITY;
  for (int g = 0; g < G; ++g) m = fmaxf(m, p[(size_t)g * ldi]);
  out[(size_t)(r % rmod) * ldo + (size_t)(r / rmod) * coloff + c] = m;
}

__global__ void __launch_bounds__(256) idx64_to_rows32_kernel(const int64_t* __restrict__ idx, size_t total,
                                                              size_t per_cloud, int N, int* __restrict__ rows) {
  for (size_t e = (size_t)blockIdx.x * 256 + threadIdx.x; e < total; e += (size_t)gridDim.x * 256)
    rows[e] = (int)(e / per_cloud) * N + (int)idx[e];
}

// Y[M,N] = act(X[M,K] W[N,K]^T + b) for skinny M (the pose MLP, model5_b.py:561-571 / :723-725: M = B <= 64 rows per
// row block).  One CTA per SK_COLS output columns and 64 rows over the WHOLE K: grid = N / 8 CTAs (128 for the first
// layer), so every layer is ONE launch with no split-K partials and no finishing pass.  X and the 8 weight rows stream
// through shared memory in 128-wide K chunks, double-buffered with cp.async (16-byte copies; the next chunk lands while
// the current one is multiplied).  Thread = (row pair, K-eighth): 2 rows x 8 columns of accumulators, 16 k per chunk;
// the eight K-eighths are summed in a fixed order (deterministic, fp32).
constexpr int SK_COLS = 8, SK_ROWS = 64, SK_KC = 128, SK_XLD = SK_KC + 4;   // +4 floats: conflict-free row reads, 16-byte rows
constexpr size_t SK_SMEM = (size_t)(2 * SK_ROWS * SK_XLD + 2 * SK_COLS * SK_KC) * sizeof(float);
__global__ void __launch_bounds__(256) skinny_linear_kernel(const float* __restrict__ X, int ldx,
                                                            const float* __restrict__ W, const float* __restrict__ bias,
                                                            int M, int N, int K, int relu, float* __restrict__ Y, int ldy) {
  extern __shared__ __align__(16) float sk_smem[];
  pdl_enter();
  float* xs = sk_smem;                                   // [2][64][SK_XLD]
  float* ws = sk_smem + 2 * SK_ROWS * SK_XLD;            // [2][8][128]
  const int tid = threadIdx.x, r2 = tid & 31, ke = tid >> 5;
  const int n0 = blockIdx.x * SK_COLS, m0 = blockIdx.y * SK_ROWS;
  const int chunks = K / SK_KC;                          // K % 128 == 0 (checked by the launcher)
  auto issue = [&](int c) {
    const int k0 = c * SK_KC;
    float* xd = xs + (c & 1) * SK_ROWS * SK_XLD;
    float* wd = ws + (c & 1) * SK_COLS * SK_KC;
    for (int e = tid; e < SK_ROWS * (SK_KC / 4); e += 256) {        // 64 rows x 32 16-byte pieces
      const int rr = e >> 5, k4 = (e & 31) * 4;
      const int row = min(m0 + rr, M - 1);                         // rows past M are computed and dropped
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(xd + rr * SK_XLD + k4)),
                   "l"(X + (size_t)row * ldx + k0 + k4) : "memory");
    }
    for (int e = tid; e < SK_COLS * (SK_KC / 4); e += 256) {
      const int nn = e >> 5, k4 = (e & 31) * 4;
      const int col = min(n0 + nn, N - 1);
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(wd + nn * SK_KC + k4)),
                   "l"(W + (size_t)col * K + k0 + k4) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  float acc[2][SK_COLS];
#pragma unroll
  for (int n = 0; n < SK_COLS; ++n) acc[0][n] = acc[1][n] = 0.f;
  issue(0);
  for (int c = 0; c < chunks; ++c) {
    if (c + 1 < chunks) {
      issue(c + 1);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
    const float* xa = xs + (c & 1) * SK_ROWS * SK_XLD + r2 * SK_XLD + ke * 16;
    const float* xb = xa + 32 * SK_XLD;
    const float* wc = ws + (c & 1) * SK_COLS * SK_KC + ke * 16;
#pragma unroll
    for (int k4 = 0; k4 < 16; k4 += 4) {
      const float4 a4 = *reinterpret_cast<const float4*>(xa + k4), b4 = *reinterpret_cast<const float4*>(xb + k4);
#pragma unroll
      for (int n = 0; n < SK_COLS; ++n) {
        const float4 w4 = *reinterpret_cast<const float4*>(wc + n * SK_KC + k4);
        acc[0][n] = fmaf(a4.x, w4.x, acc[0][n]); acc[0][n] = fmaf(a4.y, w4.y, acc[0][n]);
        acc[0][n] = fmaf(a4.z, w4.z, acc[0][n]); acc[0][n] = fmaf(a4.w, w4.w, acc[0][n]);
        acc[1][n] = fmaf(b4.x, w4.x, acc[1][n]); acc[1][n] = fmaf(b4.y, w4.y, acc[1][n]);
        acc[1][n] = fmaf(b4.z, w4.z, acc[1][n]); acc[1][n] = fmaf(b4.w, w4.w, acc[1][n]);
      }
    }
    __syncthreads();   // the buffer is refilled by the chunk after next
  }
  float* red = xs;     // [8 k-eighths][64 rows][8 cols] = 16 KB, over the (now idle) X buffers
#pragma unroll
  for (int n = 0; n < SK_COLS; ++n) {
    red[(ke * SK_ROWS + r2) * SK_COLS + n] = acc[0][n];
    red[(ke * SK_ROWS + r2 + 32) * SK_COLS + n] = acc[1][n];
  }
  __syncthreads();
  for (int e = tid; e < SK_ROWS * SK_COLS; e += 256) {
    const int rr = e >> 3, nn = e & 7;
    if (m0 + rr < M && n0 + nn < N) {
      float v = 0.f;
#pragma unroll
      for (int z = 0; z < 8; ++z) v += red[(z * SK_ROWS + rr) * SK_COLS + nn];
      if (bias) v += bias[n0 + nn];
      if (relu) v = fmaxf(v, 0.f);
      Y[(size_t)(m0 + rr) * ldy + n0 + nn] = v;
    }
  }
}

// Pose-MLP layer: one launch of skinny_linear_kernel (K % 128 == 0, 16-byte aligned rows); anything else through the
// tiled fp32 GEMM.
static int skinny_linear(const float* A, int lda, const float* W, const float* bias, int M, int N, int K,
                         int relu, float* Y, int ldy, cudaStream_t st) {
  if (K % SK_KC == 0 && lda % 4 == 0 && (((uintptr_t)A | (uintptr_t)W) & 15) == 0) {
    PZ_CUDA(cudaFuncSetAttribute(skinny_linear_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SK_SMEM));
    dim3 grid((N + SK_COLS - 1) / SK_COLS, (M + SK_ROWS - 1) / SK_ROWS);
    PZ_CUDA(launch_pdl(skinny_linear_kernel, grid, dim3(256), SK_SMEM, st, A, lda, W, bias, M, N, K, relu, Y, ldy));
    PZ_LAUNCH_CHECK();
    return 0;
  }
  GemmF32 g;
  g.A = A; g.lda = lda; g.W[0] = W; g.bias[0] = bias; g.ldw = K; g.Y = Y; g.ldy = ldy;
  g.M = M; g.N = N; g.K = K; g.relu = relu;
  return launch_gemm_f32(g, st);
}

// ----------------------------------------------------- boundary heads (model5_b.py:738-754)
// MLPLocalPre{Fpc,Rpc}: 64-64-64-64 per point, one thread per point, weights broadcast from smem.
using Mlp3W = HeadMlp3;   // (w0, b0, w1, b1, w2, b2); shared with heads_split.cu

// out[k] = act(bias[k] + W[k,:] . in) for one point per thread; W rows broadcast from smem as
// 128-bit loads, results parked in smem ([k][thread], conflict-free) so that the k loop need not be
// unrolled (a register-array destination would force full unrolling of 64 x 64 FMAs per layer).
template <int NOUT, bool RELU>
__device__ __forceinline__ void dense64_rows(const float* __restrict__ ws, const float* __restrict__ bs,
                                             const float (&in)[64], float* __restrict__ outs, int tid) {
#pragma unroll 2
  for (int k = 0; k < NOUT; ++k) {
    const float4* wr = reinterpret_cast<const float4*>(ws + k * 64);
    float v = bs[k];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      float4 ww = wr[i];
      v = fmaf(ww.x, in[i * 4 + 0], v);
      v = fmaf(ww.y, in[i * 4 + 1], v);
      v = fmaf(ww.z, in[i * 4 + 2], v);
      v = fmaf(ww.w, in[i * 4 + 3], v);
    }
    outs[k * 128 + tid] = RELU ? fmaxf(v, 0.f) : v;
  }
}

__global__ void __launch_bounds__(128) head_local_kernel(const float* __restrict__ xfeat, Mlp3W wa, Mlp3W wb,
                                                         int clouds_per_set, float* __restrict__ local) {
  extern __shared__ __align__(16) float hl_smem[];  // 3 x (64*64 + 64) weights, then [64][128] staging
  float* outs = hl_smem + 3 * 4160;
  const int tid = threadIdx.x;
  const size_t p = (size_t)blockIdx.x * 128 + tid;
  const int cloud = (int)(p / NPTS);
  const bool first = (cloud / clouds_per_set) == 0;
  const float* ws[3] = {first ? wa.w0 : wb.w0, first ? wa.w1 : wb.w1, first ? wa.w2 : wb.w2};
  const float* bs[3] = {first ? wa.b0 : wb.b0, first ? wa.b1 : wb.b1, first ? wa.b2 : wb.b2};
  for (int l = 0; l < 3; ++l) {
    for (int i = tid; i < 64 * 64; i += 128) hl_smem[l * 4160 + i] = ws[l][i];
    if (tid < 64) hl_smem[l * 4160 + 4096 + tid] = bs[l][tid];
  }
  __syncthreads();
  float a[64];
  const float4* src = reinterpret_cast<const float4*>(xfeat + p * 64);
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    float4 x = src[i];
    a[i * 4] = x.x; a[i * 4 + 1] = x.y; a[i * 4 + 2] = x.z; a[i * 4 + 3] = x.w;
  }
  dense64_rows<64, true>(hl_smem, hl_smem + 4096, a, outs, tid);
#pragma unroll
  for (int i = 0; i < 64; ++i) a[i] = outs[i * 128 + tid];
  dense64_rows<64, true>(hl_smem + 4160, hl_smem + 4160 + 4096, a, outs, tid);
#pragma unroll
  for (int i = 0; i < 64; ++i) a[i] = outs[i * 128 + tid];
  dense64_rows<64, false>(hl_smem + 2 * 4160, hl_smem + 2 * 4160 + 4096, a, outs, tid);
  float4* dst = reinterpret_cast<float4*>(local + p * 64);
#pragma unroll
  for (int i = 0; i < 16; ++i)
    dst[i] = make_float4(outs[(i * 4) * 128 + tid], outs[(i * 4 + 1) * 128 + tid], outs[(i * 4 + 2) * 128 + tid],
                         outs[(i * 4 + 3) * 128 + tid]);
}

// gbias[set][b][k] = W0_set[k, 0:64] . g[r] + b0_set[k]   (the "global" half of MLP{F,R}pcb.0), r = b, or pairs[b,1]
// when a pair list is given.  g [rows, tiles, 64]: the global feature of row r is the max over its `tiles` vectors.
__global__ void __launch_bounds__(64) seg_bias_kernel(const float* __restrict__ g, int tiles,
                                                      const int64_t* __restrict__ pairs, const float* w0a,
                                                      const float* b0a, const float* w0b, const float* b0b, int B,
                                                      float* __restrict__ gbias) {
  const int b = blockIdx.x, set = blockIdx.y, k = threadIdx.x;
  const float* w0 = set == 0 ? w0a : w0b;
  const float* b0 = set == 0 ? b0a : b0b;
  const float* gr = g + (size_t)(pairs ? pairs[2 * b + 1] : b) * tiles * 64;
  float v = b0[k];
  for (int i = 0; i < 64; ++i) {
    float gi = gr[i];
    for (int t = 1; t < tiles; ++t) gi = fmaxf(gi, gr[t * 64 + i]);
    v = fmaf(w0[k * 128 + i], gi, v);
  }
  gbias[((size_t)set * B + b) * 64 + k] = v;
}

// MLP{F,R}pcb on cat([global, local]): 128-64-32-2, logits stored as [B,2,1024] (model5_b.py:751-754).
// pairs == null: cloud c of the 2B (set = c / B, b = c % B) reads local[c].  pairs [B,2]: every cloud is a pair of
// set 0 and pair b reads local[pairs[b,0]].  Either way the bias is gbias[set][b] and the logits go to row b.
__global__ void __launch_bounds__(128) head_seg_kernel(const float* __restrict__ local, Mlp3W wa, Mlp3W wb,
                                                       const float* __restrict__ gbias, int B,
                                                       float* __restrict__ de_a, float* __restrict__ de_b,
                                                       const int64_t* __restrict__ pairs) {
  extern __shared__ __align__(16) float hs_smem[];
  float* w0s = hs_smem;            // [64][64] local half of layer 0
  float* w1s = w0s + 64 * 64;      // [32][64]
  float* gbs = w1s + 32 * 64;      // [64] per-cloud bias = global half + b0
  float* b1s = gbs + 64;           // [32]
  float* w2s = b1s + 32;           // [2][32]
  float* b2s = w2s + 64;           // [2] (+2 pad)
  float* outs = b2s + 4;           // [64][128]
  const int tid = threadIdx.x;
  const size_t p = (size_t)blockIdx.x * 128 + tid;
  const int cloud = (int)(p / NPTS);
  const int n = (int)(p - (size_t)cloud * NPTS);
  const int set = cloud / B, b = cloud - set * B;
  const Mlp3W& w = set == 0 ? wa : wb;
  for (int i = tid; i < 64 * 64; i += 128) w0s[i] = w.w0[(i >> 6) * 128 + 64 + (i & 63)];
  for (int i = tid; i < 32 * 64; i += 128) w1s[i] = w.w1[i];
  if (tid < 64) {
    w2s[tid] = w.w2[tid];
    gbs[tid] = gbias[((size_t)set * B + b) * 64 + tid];
  }
  if (tid < 32) b1s[tid] = w.b1[tid];
  if (tid < 2) b2s[tid] = w.b2[tid];
  __syncthreads();
  float a[64];
  const size_t row = pairs ? (size_t)pairs[2 * b] * NPTS + n : p;
  const float4* src = reinterpret_cast<const float4*>(local + row * 64);
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    float4 x = src[i];
    a[i * 4] = x.x; a[i * 4 + 1] = x.y; a[i * 4 + 2] = x.z; a[i * 4 + 3] = x.w;
  }
  dense64_rows<64, true>(w0s, gbs, a, outs, tid);
#pragma unroll
  for (int i = 0; i < 64; ++i) a[i] = outs[i * 128 + tid];
  dense64_rows<32, true>(w1s, b1s, a, outs, tid);
  float o0 = b2s[0], o1 = b2s[1];
#pragma unroll
  for (int k = 0; k < 32; ++k) {
    const float v = outs[k * 128 + tid];
    o0 = fmaf(w2s[k], v, o0);
    o1 = fmaf(w2s[32 + k], v, o1);
  }
  float* de = set == 0 ? de_a : de_b;
  de[((size_t)b * 2 + 0) * NPTS + n] = o0;
  de[((size_t)b * 2 + 1) * NPTS + n] = o1;
}

// ------------------------------------------------------------ se3.exp (se_math/se3.py:57-80)
__global__ void se3_exp_kernel(const float* __restrict__ x, int B, float* __restrict__ g) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float tw[6], m[16];
  for (int i = 0; i < 6; ++i) tw[i] = x[b * 6 + i];
  se3_exp_dev(tw, m);
  float* o = g + (size_t)b * 16;
  for (int i = 0; i < 16; ++i) o[i] = m[i];
}

// ------------------------------------------------ bf16 path helpers (PZ_PREC_BF16)
// One launch converts / concatenates every weight the tensor-core path needs (fp32 reference layout ->
// bf16 packs with 16-byte aligned rows).  Job y = blockIdx.y.
// to_bf16 == 2: attention-layer tile images (attention_layer_tc.cu): cols == 256, ldo = first row of the block inside
// the layer's row sequence; element (r, c) -> tile (r / 128) * 4 + c / 64, SWIZZLE_128B byte order inside the tile
struct PackJob {
  const float* src;
  void* dst;
  int ldi, rows, cols, ldo, to_bf16;
};
constexpr int MAX_PACK_JOBS = 128;
struct PackJobs {
  PackJob j[MAX_PACK_JOBS];
  int n;
};
__global__ void __launch_bounds__(256) pack_weights_kernel(const PackJobs jobs) {
  const PackJob& jb = jobs.j[blockIdx.y];
  const int total = jb.rows * jb.cols;
  for (int e = blockIdx.x * 256 + threadIdx.x; e < total; e += gridDim.x * 256) {
    const int r = e / jb.cols, c = e - r * jb.cols;
    const float v = jb.src[(size_t)r * jb.ldi + c];
    if (jb.to_bf16 == 2) {
      const int rr = r + jb.ldo, tile = (rr >> 7) * 4 + (c >> 6), tr = rr & 127, tc = c & 63;
      static_cast<__nv_bfloat16*>(jb.dst)[(size_t)tile * 8192 + tr * 64 + (((tc >> 3) ^ (tr & 7)) << 3) + (tc & 7)] =
          __float2bfloat16_rn(v);
    } else if (jb.to_bf16 == 3) {   // low half of a split-bf16 weight: v - bf16(v)
      static_cast<__nv_bfloat16*>(jb.dst)[(size_t)r * jb.ldo + c] = __float2bfloat16_rn(v - __bfloat162float(__float2bfloat16_rn(v)));
    } else if (jb.to_bf16 == 4 || jb.to_bf16 == 5) {   // split path: fp16 hi plane / lo plane (v - hi)
      const __half hi = __float2half_rn(v);
      static_cast<__half*>(jb.dst)[(size_t)r * jb.ldo + c] = jb.to_bf16 == 4 ? hi : __float2half_rn(v - __half2float(hi));
    } else if (jb.to_bf16) static_cast<__nv_bfloat16*>(jb.dst)[(size_t)r * jb.ldo + c] = __float2bfloat16_rn(v);
    else static_cast<float*>(jb.dst)[(size_t)r * jb.ldo + c] = v;
  }
}

// ======================================================================== orchestration
static StemW stem_of(const PzEncoderWeights& w) {
  return StemW{w.mlp1_w, w.mlp1_b, w.mlp2_w, w.mlp2_b, w.bn1_w, w.bn1_b, w.bn1_mean, w.bn1_var,
               w.bn2_w, w.bn2_b, w.bn2_mean, w.bn2_var};
}

static bool encoder_weights_ok(const PzEncoderWeights& w) {
  const void* const* p = reinterpret_cast<const void* const*>(&w);
  for (size_t i = 0; i < sizeof(PzEncoderWeights) / sizeof(void*); ++i)
    if (!p[i]) return false;
  return true;
}

// ---- the encoder's workspace: a common part, then the layout of the precision that runs (encoder_forward_impl).
// Common: tensors of every precision; xfeat, nx2 and fglob are replaced by the caller's outputs where it asked for them.
struct EncoderCommon { float *xfeat, *nx1, *nx2, *fglob; int *knn1r, *knn2r; };
static void carve(int C, Arena& a, EncoderCommon& s) {
  s.xfeat = a.take<float>((size_t)C * NPTS * D0);
  s.nx1 = a.take<float>((size_t)C * S1 * 3);
  s.knn1r = a.take<int>((size_t)C * S1 * KNN);
  s.nx2 = a.take<float>((size_t)C * S2 * 3);
  s.knn2r = a.take<int>((size_t)C * S2 * KNN);
  s.fglob = a.take<float>((size_t)C * 1024);
}

// fp32 path: F1 / F2 = the feature half of layer 1 of each grouped MLP, f1f and att_cat where the caller keeps no copy,
// q / k / v / r of one attention layer, the tail's 128-row tile maxima
struct Fp32Scratch { float *F1, *f1f, *F2, *att_cat, *q, *k, *v, *r, *tilemax; };
static void carve(int C, Arena& a, Fp32Scratch& s) {
  s.F1 = a.take<float>((size_t)C * NPTS * C1A);
  s.f1f = a.take<float>((size_t)C * S1 * C1B);
  s.F2 = a.take<float>((size_t)C * S1 * C2A);
  s.att_cat = a.take<float>((size_t)C * LATT * 1280);
  s.q = a.take<float>((size_t)C * LATT * 64);
  s.k = a.take<float>((size_t)C * LATT * 64);
  s.v = a.take<float>((size_t)C * LATT * CATT);
  s.r = a.take<float>((size_t)C * LATT * CATT);
  s.tilemax = a.take<float>((size_t)C * (LATT / 128) * 1024);
}

// bf16 weight pack of ONE encoder (elements): W3f[128,64] W4[128,128] W5f[256,128] W6[256,256]
// Wout[1024,1280]  4 x (20 tile images of Wqkv|Wo for the fused attention layer)
constexpr size_t WP_W3F = 0, WP_W4 = WP_W3F + 128 * 64, WP_W5F = WP_W4 + 128 * 128, WP_W6 = WP_W5F + 256 * 128,
                 WP_WOUT = WP_W6 + 256 * 256, WP_ATTIMG = WP_WOUT + 1024 * 1280, WP_STEM = WP_ATTIMG + 4 * ATTN_WIMG_ELEMS,
                 WP_TOTAL = WP_STEM + 2 * 64 * STEM_WS;   // stem: W2 hi, lo as [64, STEM_WS] images

// bf16 path: x_feature, P1 / P2 (layer 1 of each grouped MLP over the source points), f1f and att_cat in bf16; the weight
// packs of both encoders and their q|k|v biases
struct Bf16Scratch { __nv_bfloat16 *xfeat, *P1, *f1f, *P2, *att_cat, *wpack; float* bqkv; };
static void carve(int C, Arena& a, Bf16Scratch& s) {
  s.xfeat = a.take<__nv_bfloat16>((size_t)C * NPTS * D0);
  s.P1 = a.take<__nv_bfloat16>((size_t)C * NPTS * C1A);
  s.f1f = a.take<__nv_bfloat16>((size_t)C * S1 * C1B);
  s.P2 = a.take<__nv_bfloat16>((size_t)C * S1 * C2A);
  s.att_cat = a.take<__nv_bfloat16>((size_t)C * LATT * 1280);
  s.wpack = a.take<__nv_bfloat16>(2 * WP_TOTAL);
  s.bqkv = a.take<float>(2 * 4 * 384);
}

// split path: fp16 planes of ONE encoder (elements per plane): W3f[128,64] W4[128,128] W5f[256,128] W6[256,256]
// 4 x (Wqk[128,256] Wv[256,256] Wo[256,256]) Wout[1024,1280]; planes at wpack + ((e * 2 + plane) * WS_TOTAL)
constexpr size_t WS_W3F = 0, WS_W4 = WS_W3F + 128 * 64, WS_W5F = WS_W4 + 128 * 128, WS_W6 = WS_W5F + 256 * 128,
                 WS_ATT = WS_W6 + 256 * 256, WS_ATT_STRIDE = 128 * 256 + 2 * 256 * 256, WS_WOUT = WS_ATT + 4 * WS_ATT_STRIDE,
                 WS_TOTAL = WS_WOUT + 1024 * 1280;

// split path: every 16-bit tensor is a pair of same-shaped fp16 planes [hi, lo], stored as the raw 16-bit type TcGemm and
// AttnSplit take.  P (layer 1 over the source points) and Q = W1[:,0:3] c of each grouped MLP stay fp32.  The chained
// attention launches read one q|k / v^T set while they write the next layer's into the other; r stays on chip (fused
// out-projection) and has no buffer.
typedef __nv_bfloat16 h16;
struct SplitScratch {
  h16 *xfeat[2], *f1f[2], *att_cat[2];   // [plane]
  h16 *qk[2][2], *vT[2][2];              // [set][plane]: q|k [C*256, 128], v^T [C][256 ch][256 tokens]
  float *P1, *Q1, *P2, *Q2;
  int* flags;                            // [3][C] hand-over counters of the chained attention launches
  float* tilemax;                        // [C*2, 1024] the tail's 128-row tile maxima
  h16* wpack;
  float* bqkv;
};
static void carve(int C, Arena& a, SplitScratch& s) {
  for (int pl = 0; pl < 2; ++pl) {
    s.xfeat[pl] = a.take<h16>((size_t)C * NPTS * D0);
    s.f1f[pl] = a.take<h16>((size_t)C * S1 * C1B);
    s.att_cat[pl] = a.take<h16>((size_t)C * LATT * 1280);
    for (int set = 0; set < 2; ++set) {
      s.qk[set][pl] = a.take<h16>((size_t)C * LATT * 128);
      s.vT[set][pl] = a.take<h16>((size_t)C * LATT * CATT);
    }
  }
  s.P1 = a.take<float>((size_t)C * NPTS * C1A);
  s.Q1 = a.take<float>((size_t)C * S1 * C1A);
  s.P2 = a.take<float>((size_t)C * S1 * C2A);
  s.Q2 = a.take<float>((size_t)C * S2 * C2A);
  s.flags = a.take<int>((size_t)3 * C);
  s.tilemax = a.take<float>((size_t)C * (LATT / 128) * 1024);
  s.wpack = a.take<h16>(4 * WS_TOTAL);
  s.bqkv = a.take<float>(2 * 4 * 384);
}

// The geometry of a forward -- FPS, kNN and, on the split path, the centre projection Q of each grouped MLP, for both
// stages -- as one launch (geometry.cu: geometry_c2_kernel).  Q1 / Q2 null: no centre projections.
static_assert(NPTS == 1024 && S1 == 512 && S2 == 256 && KNN == 32, "launch_encoder_geometry covers this shape only");
static int encoder_geometry(const PzEncoderWeights& wa, const PzEncoderWeights& wb, int B, int C, const float* xyz,
                            const int64_t* start1, const int64_t* start2, const PzEncoderOutputs& o, const EncoderCommon& c,
                            float* Q1, float* Q2, cudaStream_t st) {
  EncoderGeometry g;
  g.xyz = xyz; g.start1 = start1; g.start2 = start2;
  g.fps1 = o.fps1; g.knn1 = o.knn1; g.fps2 = o.fps2; g.knn2 = o.knn2;
  g.nx1 = c.nx1; g.nx2 = c.nx2; g.knn1r = c.knn1r; g.knn2r = c.knn2r;
  g.Q1 = Q1; g.Q2 = Q2;
  g.w1[0] = wa.mlp3_w; g.w1[1] = wb.mlp3_w; g.ldw1 = 3 + D0;
  g.w2[0] = wa.mlp5_w; g.w2[1] = wb.mlp5_w; g.ldw2 = 3 + C1B;
  g.clouds_per_set = B;
  return launch_encoder_geometry(g, C, st);
}

// ---------------------------------------------------------------------------------------------
// bf16 path: every dense layer on tcgen05 (gemm_tc.cu), geometry + softmax in fp32.
// Layer 1 of each grouped MLP is split as  W1 [xyz_j - c_s ; f_j] + b1 = P_j - Q_s  with
// P = f W1[:,3:]^T + b1 + W1[:,0:3] xyz_j (one GEMM over the SOURCE points, bf16 out) and
// Q = W1[:,0:3] c_s (per centroid); the layer-2 GEMM gathers relu(P_j - Q_s) straight into its
// shared-memory operand and max-pools over the 32 neighbours in its epilogue.
// ---------------------------------------------------------------------------------------------
// runs on the caller's stream right after the stem: work that only needs x_feature (the boundary heads of predict5)
// fills the time the stream would otherwise spend waiting for the stage-1 geometry
using AfterStem = std::function<int(const float* xfeat)>;

static int encoder_forward_bf16(const PzEncoderWeights* w, int E, int B, const float* xyz, const int64_t* start1,
                                const int64_t* start2, const PzEncoderOutputs& o, const EncoderCommon& c,
                                const Bf16Scratch& s, const AfterStem* after_stem, bool reuse_pack, cudaStream_t st) {
  const int C = E * B;
  const PzEncoderWeights& wa = w[0];
  const PzEncoderWeights& wb = w[E - 1];

  // ---- weights -> bf16 packs (one launch, ~8 MB read).  The pack lives in the caller's workspace; a caller that
  // knows the weights are unchanged since its previous call may say so (PZ_FLAG_REUSE_PACKS) and skip it.
  if (!reuse_pack) {
    PackJobs jobs;
    int n = 0;
    auto add = [&](const float* src, int ldi, int rows, int cols, void* dst, int ldo, int bf) {
      if (n < MAX_PACK_JOBS) jobs.j[n] = PackJob{src, dst, ldi, rows, cols, ldo, bf};
      ++n;
    };
    for (int e = 0; e < E; ++e) {
      const PzEncoderWeights& we = w[e];
      __nv_bfloat16* wp = s.wpack + (size_t)e * WP_TOTAL;
      add(we.mlp3_w + 3, 3 + D0, C1A, D0, wp + WP_W3F, D0, 1);
      add(we.mlp4_w, C1A, C1B, C1A, wp + WP_W4, C1A, 1);
      add(we.mlp5_w + 3, 3 + C1B, C2A, C1B, wp + WP_W5F, C1B, 1);
      add(we.mlp6_w, C2A, C2B, C2A, wp + WP_W6, C2A, 1);
      for (int l = 0; l < 4; ++l) {
        __nv_bfloat16* wi = wp + WP_ATTIMG + (size_t)l * ATTN_WIMG_ELEMS;
        add(we.q_w[l], CATT, 64, CATT, wi, 0, 2);
        add(we.k_w[l], CATT, 64, CATT, wi, 64, 2);
        add(we.v_w[l], CATT, CATT, CATT, wi, 128, 2);
        add(we.o_w[l], CATT, CATT, CATT, wi, 384, 2);
        float* bq = s.bqkv + ((size_t)e * 4 + l) * 384;
        add(we.q_b[l], 64, 1, 64, bq, 64, 0);
        add(we.k_b[l], 64, 1, 64, bq + 64, 64, 0);
        add(we.v_b[l], CATT, 1, CATT, bq + 128, CATT, 0);
      }
      add(we.out_w, 1280, 1024, 1280, wp + WP_WOUT, 1280, 1);
      add(we.mlp2_w, 64, 64, 64, wp + WP_STEM, STEM_WS, 1);
      add(we.mlp2_w, 64, 64, 64, wp + WP_STEM + 64 * STEM_WS, STEM_WS, 3);
    }
    PZ_REQUIRE(n <= MAX_PACK_JOBS, PZ_ERR_ARG, "encoder: %d weight pack jobs exceed the table", n);
    jobs.n = n;
    pack_weights_kernel<<<dim3(64, n), 256, 0, st>>>(jobs);
    PZ_LAUNCH_CHECK();
    prof_mark("pack_weights_bf16", st);
  }
  const __nv_bfloat16* wpa = s.wpack;
  const __nv_bfloat16* wpb = s.wpack + (size_t)(E - 1) * WP_TOTAL;

  // ---- geometry (FPS -> kNN, both stages) depends on coordinates only: it runs on the side stream while the feature
  // chain (stem, layer-1 GEMMs) runs on the caller's stream.
  SideStream* ss = nullptr;
  PZ_TRY(side_stream(&ss, st));
  const bool serial = prof_serial();
  cudaStream_t sg = serial ? st : ss->stream;
  const int gl = serial ? 0 : 1;   // profiler lane of the geometry marks
  PZ_CUDA(cudaEventRecord(ss->fork, st));
  PZ_CUDA(cudaStreamWaitEvent(sg, ss->fork, 0));
  prof_mark("_side_begin", sg, gl);
  PZ_TRY(encoder_geometry(wa, wb, B, C, xyz, start1, start2, o, c, nullptr, nullptr, sg));
  prof_mark("geometry", sg, gl);
  PZ_CUDA(cudaEventRecord(ss->join, sg));

  PZ_CUDA(cudaFuncSetAttribute(stem_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)STEM_TC_SMEM));
  stem_tc_kernel<false><<<C * NPTS / (128 * HD_REPS), 128, STEM_TC_SMEM, st>>>(xyz, stem_of(wa), stem_of(wb), wpa + WP_STEM,
                                                                          wpb + WP_STEM, B, HD_REPS, c.xfeat, s.xfeat, nullptr);
  PZ_LAUNCH_CHECK();
  prof_mark("stem", st);
  {
    TcGemm g;  // P1 = x_feature W3[:,3:]^T + b3 + W3[:,0:3] xyz
    g.X = s.xfeat; g.ldx = D0; g.W[0] = wpa + WP_W3F; g.W[1] = wpb + WP_W3F; g.ldw = D0;
    g.bias[0] = wa.mlp3_b; g.bias[1] = wb.mlp3_b; g.rows_per_wset = B * NPTS; g.M = C * NPTS; g.Nout = C1A; g.K = D0;
    g.Yb = s.P1; g.ldyb = C1A; g.xyz = xyz; g.W1x[0] = wa.mlp3_w; g.W1x[1] = wb.mlp3_w; g.ldw1x = 3 + D0;
    PZ_TRY(launch_tc_rowgemm(g, st));
    prof_mark("sg1_layer1", st);
  }
  if (after_stem) PZ_TRY((*after_stem)(c.xfeat));
  PZ_CUDA(cudaStreamWaitEvent(st, ss->join, 0));   // the geometry of both stages is done (side stream joined)
  prof_mark("_wait_geometry", st);
  {
    TcGemm g;  // f1f = max_k relu(W4 relu(P1[j] - Q1[s]) + b4)
    g.X = s.P1; g.ldx = C1A; g.rows = c.knn1r; g.centers = c.nx1; g.W1x[0] = wa.mlp3_w; g.W1x[1] = wb.mlp3_w; g.ldw1x = 3 + D0; g.W[0] = wpa + WP_W4; g.W[1] = wpb + WP_W4; g.ldw = C1A;
    g.bias[0] = wa.mlp4_b; g.bias[1] = wb.mlp4_b; g.rows_per_wset = B * S1 * KNN; g.M = C * S1 * KNN; g.Nout = C1B;
    g.K = C1A; g.epi = 1; g.relu = 1; g.Yf = o.f1f; g.ldyf = C1B; g.Yb = s.f1f; g.ldyb = C1B;
    PZ_TRY(launch_tc_gemm(g, st));
    prof_mark("sg1_gather_layer2_maxpool", st);
  }
  {
    TcGemm g;  // P2 = f1f W5[:,3:]^T + b5 + W5[:,0:3] x1
    g.X = s.f1f; g.ldx = C1B; g.W[0] = wpa + WP_W5F; g.W[1] = wpb + WP_W5F; g.ldw = C1B;
    g.bias[0] = wa.mlp5_b; g.bias[1] = wb.mlp5_b; g.rows_per_wset = B * S1; g.M = C * S1; g.Nout = C2A; g.K = C1B;
    g.Yb = s.P2; g.ldyb = C2A; g.xyz = c.nx1; g.W1x[0] = wa.mlp5_w; g.W1x[1] = wb.mlp5_w; g.ldw1x = 3 + C1B;
    PZ_TRY(launch_tc_rowgemm(g, st));
    prof_mark("sg2_layer1", st);
  }
  __nv_bfloat16* cat_b = s.att_cat;             // [C*256, 1280] bf16: cat(att1..att4, f2f)
  float* cat_f = o.att_cat;                     // fp32 copy only when the caller asks for it
  {
    TcGemm g;
    g.X = s.P2; g.ldx = C2A; g.rows = c.knn2r; g.centers = c.nx2; g.W1x[0] = wa.mlp5_w; g.W1x[1] = wb.mlp5_w; g.ldw1x = 3 + C1B; g.W[0] = wpa + WP_W6; g.W[1] = wpb + WP_W6; g.ldw = C2A;
    g.bias[0] = wa.mlp6_b; g.bias[1] = wb.mlp6_b; g.rows_per_wset = B * S2 * KNN; g.M = C * S2 * KNN; g.Nout = C2B;
    g.K = C2A; g.epi = 1; g.relu = 1; g.Yb = cat_b + 4 * CATT; g.ldyb = 1280;
    if (cat_f) { g.Yf = cat_f + 4 * CATT; g.ldyf = 1280; }
    else if (o.f2f) { g.Yf = o.f2f; g.ldyf = CATT; }
    PZ_TRY(launch_tc_gemm(g, st));
    prof_mark("sg2_gather_layer2_maxpool", st);
  }

  // ---- 4 x offset attention
  const int rows = C * LATT;
  {   // the four layers of a cloud in one launch: nothing but the layer inputs / outputs touches HBM
    AttnLayerTc p;
    p.nlayers = 4;
    p.x = cat_b + 4 * CATT; p.ldx = 1280;
    p.wimg[0] = wpa + WP_ATTIMG; p.wimg[1] = wpb + WP_ATTIMG;
    p.bqkv[0] = s.bqkv; p.bqkv[1] = s.bqkv + (size_t)(E - 1) * 4 * 384;
    for (int l = 0; l < 4; ++l) {
      p.bo[0][l] = wa.o_b[l]; p.bo[1][l] = wb.o_b[l];
      p.attn_mode[l] = o.attention ? (l == 0 ? 1 : (l == 3 ? 3 : 2)) : 0;
    }
    p.clouds_per_set = B; p.yb = cat_b; p.ldyb = 1280; p.yb_layer_stride = CATT;
    if (cat_f) { p.yf = cat_f; p.ldyf = 1280; p.yf_layer_stride = CATT; }
    p.attn = o.attention;
    PZ_TRY(launch_attention_layer_tc(p, C, st));
    prof_mark("attn_layer_fused", st);
  }
  // ---- tail
  TcGemm g;
  g.X = cat_b; g.ldx = 1280; g.W[0] = wpa + WP_WOUT; g.W[1] = wpb + WP_WOUT; g.ldw = 1280;
  g.bias[0] = wa.out_b; g.bias[1] = wb.out_b; g.rows_per_wset = B * LATT; g.M = rows; g.Nout = 1024; g.K = 1280;
  if (o.out) {
    g.Yf = o.out; g.ldyf = 1024;
    PZ_TRY(launch_tc_gemm(g, st));
    prof_mark("tail_linear", st);
    rowblock_max_kernel<<<dim3(4, C), 256, 0, st>>>(o.out, 1024, LATT, 1024, C, C, 0, c.fglob, 1024);
    PZ_LAUNCH_CHECK();
    prof_mark("tail_point_max", st);
  } else {
    g.epi = 2; g.Yf = c.fglob; g.ldyf = 1024;   // one 256-row tile == one cloud: max over its rows in the epilogue
    PZ_TRY(launch_tc_gemm(g, st));
    prof_mark("tail_linear_maxpool", st);
  }
  return 0;
}


// ---------------------------------------------------------------------------------------------
// split path (PZ_PREC_SPLIT): the bf16 path's dataflow with every tensor-core operand as fp16 hi / lo planes and
// every product as three MMAs (gemm_split.cu, attention_split.cu) -- the fp32 tolerances at tensor-core speed.
// P = layer 1 over the source points and Q = W1[:,0:3] c stay fp32 in HBM; the gather GEMM forms relu(P_j - Q_s) in
// fp32 registers before splitting it.
// ---------------------------------------------------------------------------------------------
static int encoder_forward_split(const PzEncoderWeights* w, int E, int B, const float* xyz, const int64_t* start1,
                                 const int64_t* start2, const PzEncoderOutputs& o, const EncoderCommon& c,
                                 const SplitScratch& s, const AfterStem* after_stem, bool reuse_pack, cudaStream_t st) {
  const int C = E * B;
  const PzEncoderWeights& wa = w[0];
  const PzEncoderWeights& wb = w[E - 1];

  if (!reuse_pack) {
    PackJobs jobs;
    int n = 0;
    auto add = [&](const float* src, int ldi, int rows, int cols, void* dst, int ldo, int mode) {
      if (n < MAX_PACK_JOBS) jobs.j[n] = PackJob{src, dst, ldi, rows, cols, ldo, mode};
      ++n;
    };
    for (int e = 0; e < E; ++e) {
      const PzEncoderWeights& we = w[e];
      for (int pl = 0; pl < 2; ++pl) {
        h16* wp = s.wpack + (size_t)(e * 2 + pl) * WS_TOTAL;
        const int mode = 4 + pl;
        add(we.mlp3_w + 3, 3 + D0, C1A, D0, wp + WS_W3F, D0, mode);
        add(we.mlp4_w, C1A, C1B, C1A, wp + WS_W4, C1A, mode);
        add(we.mlp5_w + 3, 3 + C1B, C2A, C1B, wp + WS_W5F, C1B, mode);
        add(we.mlp6_w, C2A, C2B, C2A, wp + WS_W6, C2A, mode);
        for (int l = 0; l < 4; ++l) {
          h16* wl = wp + WS_ATT + (size_t)l * WS_ATT_STRIDE;
          add(we.q_w[l], CATT, 64, CATT, wl, CATT, mode);
          add(we.k_w[l], CATT, 64, CATT, wl + 64 * CATT, CATT, mode);
          add(we.v_w[l], CATT, CATT, CATT, wl + 128 * CATT, CATT, mode);
          add(we.o_w[l], CATT, CATT, CATT, wl + 384 * CATT, CATT, mode);
        }
        add(we.out_w, 1280, 1024, 1280, wp + WS_WOUT, 1280, mode);
      }
      for (int l = 0; l < 4; ++l) {
        float* bq = s.bqkv + ((size_t)e * 4 + l) * 384;
        add(we.q_b[l], 64, 1, 64, bq, 64, 0);
        add(we.k_b[l], 64, 1, 64, bq + 64, 64, 0);
        add(we.v_b[l], CATT, 1, CATT, bq + 128, CATT, 0);
      }
    }
    PZ_REQUIRE(n <= MAX_PACK_JOBS, PZ_ERR_ARG, "encoder: %d weight pack jobs exceed the table", n);
    jobs.n = n;
    pack_weights_kernel<<<dim3(64, n), 256, 0, st>>>(jobs);
    PZ_LAUNCH_CHECK();
    prof_mark("pack_weights_split", st);
  }
  const h16* wp_[2][2] = {{s.wpack, s.wpack + WS_TOTAL},
                          {s.wpack + (size_t)(E - 1) * 2 * WS_TOTAL, s.wpack + ((size_t)(E - 1) * 2 + 1) * WS_TOTAL}};
  auto set_w = [&](TcGemm& g, size_t off) {
    g.W[0] = wp_[0][0] + off; g.Wlo[0] = wp_[0][1] + off; g.W[1] = wp_[1][0] + off; g.Wlo[1] = wp_[1][1] + off;
  };

  // the attention launches' hand-over counters (see the attention block): zeroed here, where no kernel-to-kernel link of the
  // programmatic launch chain is broken by the memset node
  PZ_CUDA(cudaMemsetAsync(s.flags, 0, (size_t)3 * C * sizeof(int), st));

  // ---- geometry (FPS, kNN and the centre projections Q1 / Q2, both stages, one launch): ahead of the feature chain on the
  // caller's stream.
  // ONE chain: every GEMM CTA of this path fills an SM (shared memory), so a geometry kernel on a second stream does not
  // share SMs with them, it delays some of the CTAs of a persistent GEMM and the whole launch waits for those (eager
  // forward 1.70 ms with a side stream, 1.59 without, 1.51 with programmatic dependent launch on the one chain; the
  // 4-stream graph schedule 1.39 vs 1.37 ms per step).
  prof_mark("_side_begin", st);
  static_assert(C1A == 128 && C2A == 256, "geometry_c2_kernel writes Q1 / Q2 rows of 128 / 256 channels");
  PZ_TRY(encoder_geometry(wa, wb, B, C, xyz, start1, start2, o, c, s.Q1, s.Q2, st));
  prof_mark("geometry", st);

  // ---- feature chain
  // stem: layer 2 as a split-fp16 mma.sync product (x_feature within ~1e-6 of the fp32 stem), the fp16 hi / lo planes of
  // x_feature written by the same kernel (C * 1024 points always tile by 128 * HD_REPS)
  PZ_CUDA(cudaFuncSetAttribute(stem_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)STEM_TC_SMEM));
  PZ_CUDA(launch_pdl(stem_tc_kernel<true>, dim3(C * NPTS / (128 * HD_REPS)), dim3(128), STEM_TC_SMEM, st, xyz, stem_of(wa),
                     stem_of(wb), (const __nv_bfloat16*)nullptr, (const __nv_bfloat16*)nullptr, B, HD_REPS, c.xfeat,
                     s.xfeat[0], reinterpret_cast<__half*>(s.xfeat[1])));
  PZ_LAUNCH_CHECK();
  prof_mark("stem", st);
  {
    TcGemm g;  // P1 = x_feature W3[:,3:]^T + b3 + W3[:,0:3] xyz   (fp32 out)
    g.X = s.xfeat[0]; g.Xlo = s.xfeat[1]; g.ldx = D0; set_w(g, WS_W3F); g.ldw = D0;
    g.bias[0] = wa.mlp3_b; g.bias[1] = wb.mlp3_b; g.rows_per_wset = B * NPTS; g.M = C * NPTS; g.Nout = C1A; g.K = D0;
    g.Yf = s.P1; g.ldyf = C1A; g.xyz = xyz; g.W1x[0] = wa.mlp3_w; g.W1x[1] = wb.mlp3_w; g.ldw1x = 3 + D0;
    PZ_TRY(launch_split_rowgemm(g, st));
    prof_mark("sg1_layer1", st);
  }
  if (after_stem) PZ_TRY((*after_stem)(c.xfeat));
  prof_mark("_wait_geometry1", st);
  {
    TcGemm g;  // f1f = max_k relu(W4 relu(P1[j] - Q1[s]) + b4)
    g.Xf = s.P1; g.ldx = C1A; g.Qf = s.Q1; g.rows = c.knn1r; set_w(g, WS_W4); g.ldw = C1A;
    g.bias[0] = wa.mlp4_b; g.bias[1] = wb.mlp4_b; g.rows_per_wset = B * S1 * KNN; g.M = C * S1 * KNN; g.Nout = C1B;
    g.K = C1A; g.epi = 1; g.relu = 1; g.Yf = o.f1f; g.ldyf = C1B; g.Yb = s.f1f[0]; g.Yblo = s.f1f[1]; g.ldyb = C1B;
    PZ_TRY(launch_split_gather(g, st));
    prof_mark("sg1_gather_layer2_maxpool", st);
  }
  {
    TcGemm g;  // P2 = f1f W5[:,3:]^T + b5 + W5[:,0:3] x1
    g.X = s.f1f[0]; g.Xlo = s.f1f[1]; g.ldx = C1B; set_w(g, WS_W5F); g.ldw = C1B;
    g.bias[0] = wa.mlp5_b; g.bias[1] = wb.mlp5_b; g.rows_per_wset = B * S1; g.M = C * S1; g.Nout = C2A; g.K = C1B;
    g.Yf = s.P2; g.ldyf = C2A; g.xyz = c.nx1; g.W1x[0] = wa.mlp5_w; g.W1x[1] = wb.mlp5_w; g.ldw1x = 3 + C1B;
    PZ_TRY(launch_split_rowgemm(g, st));
    prof_mark("sg2_layer1", st);
  }
  prof_mark("_wait_geometry2", st);
  float* cat_f = o.att_cat;
  {
    TcGemm g;
    g.Xf = s.P2; g.ldx = C2A; g.Qf = s.Q2; g.rows = c.knn2r; set_w(g, WS_W6); g.ldw = C2A;
    g.bias[0] = wa.mlp6_b; g.bias[1] = wb.mlp6_b; g.rows_per_wset = B * S2 * KNN; g.M = C * S2 * KNN; g.Nout = C2B;
    g.K = C2A; g.epi = 1; g.relu = 1; g.Yb = s.att_cat[0] + 4 * CATT; g.Yblo = s.att_cat[1] + 4 * CATT; g.ldyb = 1280;
    if (cat_f) { g.Yf = cat_f + 4 * CATT; g.ldyf = 1280; }
    else if (o.f2f) { g.Yf = o.f2f; g.ldyf = CATT; }
    PZ_TRY(launch_split_gather(g, st));
    prof_mark("sg2_gather_layer2_maxpool", st);
  }

  // ---- 4 x offset attention
  const int rows = C * LATT;
  // the out-projection  out = x + relu(Wo r + bo)  runs inside the attention kernel (r never leaves the SM: 67 MB of HBM
  // traffic and one launch per layer less), and so do the NEXT layer's q|k|v projections of the same rows (chained: two
  // more launches per layer less); q|k and v^T planes then alternate between two buffer sets, because the CTAs of a launch
  // still read the current ones.  Chained launches hand over per cloud (AttnSplit::dep_flags, 3 x C counters).
  for (int l = 0; l < 4; ++l) {
    const size_t xoff = l == 0 ? 4 * CATT : (size_t)(l - 1) * CATT;
    const size_t wl = WS_ATT + (size_t)l * WS_ATT_STRIDE;
    const int cur = l & 1;
    if (l == 0) {
      TcGemm gq;  // [q | k] = x Wqk^T + b
      gq.X = s.att_cat[0] + xoff; gq.Xlo = s.att_cat[1] + xoff; gq.ldx = 1280; set_w(gq, wl); gq.ldw = CATT;
      gq.bias[0] = s.bqkv + (size_t)l * 384; gq.bias[1] = s.bqkv + ((size_t)(E - 1) * 4 + l) * 384;
      gq.rows_per_wset = B * LATT; gq.M = rows; gq.Nout = 128; gq.K = CATT; gq.Yb = s.qk[cur][0]; gq.Yblo = s.qk[cur][1]; gq.ldyb = 128;
      PZ_TRY(launch_split_rowgemm(gq, st));
      TcGemm gv = gq;  // v^T per cloud (K-major operand of P v)
      set_w(gv, wl + 128 * CATT); gv.bias[0] = gq.bias[0] + 128; gv.bias[1] = gq.bias[1] + 128;
      gv.Nout = CATT; gv.Yb = nullptr; gv.Yblo = nullptr; gv.YT = s.vT[cur][0]; gv.YTlo = s.vT[cur][1]; gv.t_rows = LATT;
      PZ_TRY(launch_split_rowgemm(gv, st));
      prof_mark("attn_qkv_proj", st);
    }
    AttnSplit ap;
    ap.qk_hi = s.qk[cur][0]; ap.qk_lo = s.qk[cur][1]; ap.vT_hi = s.vT[cur][0]; ap.vT_lo = s.vT[cur][1];
    ap.x_hi = s.att_cat[0] + xoff; ap.x_lo = s.att_cat[1] + xoff; ap.ldx = 1280;
    ap.attn = o.attention; ap.attn_mode = o.attention ? (l == 0 ? 1 : (l == 3 ? 3 : 2)) : 0;
    ap.wo_hi[0] = wp_[0][0] + wl + 384 * CATT; ap.wo_lo[0] = wp_[0][1] + wl + 384 * CATT;
    ap.wo_hi[1] = wp_[1][0] + wl + 384 * CATT; ap.wo_lo[1] = wp_[1][1] + wl + 384 * CATT;
    ap.bo[0] = wa.o_b[l]; ap.bo[1] = wb.o_b[l]; ap.clouds_per_set = B;
    ap.y_hi = s.att_cat[0] + (size_t)l * CATT; ap.y_lo = s.att_cat[1] + (size_t)l * CATT; ap.ldy = 1280;
    if (cat_f) { ap.yf = cat_f + (size_t)l * CATT; ap.ldyf = 1280; }
    if (l < 3) {   // the next layer's projections of these rows
      const size_t wn = WS_ATT + (size_t)(l + 1) * WS_ATT_STRIDE;
      ap.wqkv_hi[0] = wp_[0][0] + wn; ap.wqkv_lo[0] = wp_[0][1] + wn; ap.wqkv_hi[1] = wp_[1][0] + wn; ap.wqkv_lo[1] = wp_[1][1] + wn;
      ap.bqkv[0] = s.bqkv + (size_t)(l + 1) * 384; ap.bqkv[1] = s.bqkv + ((size_t)(E - 1) * 4 + l + 1) * 384;
      ap.qk2_hi = s.qk[cur ^ 1][0]; ap.qk2_lo = s.qk[cur ^ 1][1]; ap.vT2_hi = s.vT[cur ^ 1][0]; ap.vT2_lo = s.vT[cur ^ 1][1];
      ap.sig_flags = s.flags + (size_t)l * C;
    }
    if (l > 0) ap.dep_flags = s.flags + (size_t)(l - 1) * C;
    PZ_TRY(launch_attention_split(ap, C, st));
    prof_mark("attn_softmax_av", st);
  }
  // ---- tail: Linear(1280, 1024), then the max over the 256 points of a cloud
  TcGemm g;
  g.X = s.att_cat[0]; g.Xlo = s.att_cat[1]; g.ldx = 1280; set_w(g, WS_WOUT); g.ldw = 1280;
  g.bias[0] = wa.out_b; g.bias[1] = wb.out_b; g.rows_per_wset = B * LATT; g.M = rows; g.Nout = 1024; g.K = 1280;
  if (o.out) { g.Yf = o.out; g.ldyf = 1024; }
  g.Ymax = s.tilemax; g.ldmax = 1024;           // per 128-row tile column maxima: two tiles per cloud
  PZ_TRY(launch_split_rowgemm(g, st));
  prof_mark("tail_linear_maxpool", st);
  PZ_CUDA(launch_pdl(rowblock_max_kernel, dim3(4, C), dim3(256), 0, st, (const float*)s.tilemax, 1024, LATT / 128, 1024, C, C, 0,
                     c.fglob, 1024));
  PZ_LAUNCH_CHECK();
  prof_mark("tail_point_max", st);
  return 0;
}

// fp32 path (PZ_PREC_FP32): every tensor and product in fp32 on the CUDA cores (stem_kernel, gemm_f32.cu)
static int encoder_forward_fp32(const PzEncoderWeights* w, int E, int B, const float* xyz, const int64_t* start1,
                                const int64_t* start2, const PzEncoderOutputs& o, const EncoderCommon& c,
                                const Fp32Scratch& s, const AfterStem* after_stem, cudaStream_t st) {
  const int C = E * B;
  const PzEncoderWeights& wa = w[0];
  const PzEncoderWeights& wb = w[E - 1];
  float* f1f = o.f1f ? o.f1f : s.f1f;
  float* att_cat = o.att_cat ? o.att_cat : s.att_cat;

  // stem: Linear(3,64)+BN+ReLU, Linear(64,64)+BN+ReLU -> x_feature [C,1024,64]
  stem_kernel<<<C * NPTS / 128, 128, 0, st>>>(xyz, stem_of(wa), stem_of(wb), B, c.xfeat);
  PZ_LAUNCH_CHECK();
  prof_mark("stem", st);
  if (after_stem) PZ_TRY((*after_stem)(c.xfeat));

  // ---- geometry of both stages: FPS 1024->512, kNN 32, FPS 512->256 on the stage-1 centroids, kNN 32
  PZ_TRY(encoder_geometry(wa, wb, B, C, xyz, start1, start2, o, c, nullptr, nullptr, st));
  prof_mark("geometry", st);
  // ---- stage 1: grouped MLP 67->128->128, max over K
  {
    GemmF32 g;  // F1 = x_feature * mlp3.weight[:, 3:]^T   (bias + xyz part are added per neighbour)
    g.A = c.xfeat; g.lda = D0; g.W[0] = wa.mlp3_w + 3; g.W[1] = wb.mlp3_w + 3; g.ldw = 3 + D0;
    g.rows_per_wset = B * NPTS; g.Y = s.F1; g.ldy = C1A; g.M = C * NPTS; g.N = C1A; g.K = D0;
    PZ_TRY(launch_gemm_f32(g, st));
    prof_mark("sg1_layer1", st);
  }
  {
    GemmF32 g;
    g.A = s.F1; g.lda = C1A; g.rows = c.knn1r; g.xyz = xyz; g.centers = c.nx1;
    g.W1[0] = wa.mlp3_w; g.W1[1] = wb.mlp3_w; g.b1[0] = wa.mlp3_b; g.b1[1] = wb.mlp3_b; g.ldw1 = 3 + D0;
    g.W[0] = wa.mlp4_w; g.W[1] = wb.mlp4_w; g.bias[0] = wa.mlp4_b; g.bias[1] = wb.mlp4_b; g.ldw = C1A;
    g.rows_per_wset = B * S1 * KNN; g.Y = f1f; g.ldy = C1B; g.M = C * S1 * KNN; g.N = C1B; g.K = C1A;
    g.relu = 1; g.group = 32;
    PZ_TRY(launch_gemm_f32(g, st));
    prof_mark("sg1_gather_layer2_maxpool", st);
  }
  // ---- stage 2: grouped MLP 131->256->256
  {
    GemmF32 g;
    g.A = f1f; g.lda = C1B; g.W[0] = wa.mlp5_w + 3; g.W[1] = wb.mlp5_w + 3; g.ldw = 3 + C1B;
    g.rows_per_wset = B * S1; g.Y = s.F2; g.ldy = C2A; g.M = C * S1; g.N = C2A; g.K = C1B;
    PZ_TRY(launch_gemm_f32(g, st));
    prof_mark("sg2_layer1", st);
  }
  float* f2f_slot = att_cat + 4 * CATT;  // cat([att1..att4, f2f]) (model5_b.py:467,472): f2f is columns 1024..1279
  {
    GemmF32 g;
    g.A = s.F2; g.lda = C2A; g.rows = c.knn2r; g.xyz = c.nx1; g.centers = c.nx2;
    g.W1[0] = wa.mlp5_w; g.W1[1] = wb.mlp5_w; g.b1[0] = wa.mlp5_b; g.b1[1] = wb.mlp5_b; g.ldw1 = 3 + C1B;
    g.W[0] = wa.mlp6_w; g.W[1] = wb.mlp6_w; g.bias[0] = wa.mlp6_b; g.bias[1] = wb.mlp6_b; g.ldw = C2A;
    g.rows_per_wset = B * S2 * KNN; g.Y = f2f_slot; g.ldy = 1280; g.M = C * S2 * KNN; g.N = C2B; g.K = C2A;
    g.relu = 1; g.group = 32;
    PZ_TRY(launch_gemm_f32(g, st));
    prof_mark("sg2_gather_layer2_maxpool", st);
  }

  // ---- 4 x offset attention (model5_b.py:92-101); layer i writes att_cat[:, i*256:(i+1)*256]
  const int rows = C * LATT;
  for (int l = 0; l < 4; ++l) {
    const float* x = l == 0 ? f2f_slot : att_cat + (l - 1) * CATT;
    auto proj = [&](const float* w0, const float* w1, const float* b0, const float* b1, int N, float* y) {
      GemmF32 g;
      g.A = x; g.lda = 1280; g.W[0] = w0; g.W[1] = w1; g.bias[0] = b0; g.bias[1] = b1; g.ldw = CATT;
      g.rows_per_wset = B * LATT; g.Y = y; g.ldy = N; g.M = rows; g.N = N; g.K = CATT;
      return launch_gemm_f32(g, st);
    };
    PZ_TRY(proj(wa.q_w[l], wb.q_w[l], wa.q_b[l], wb.q_b[l], 64, s.q));
    PZ_TRY(proj(wa.k_w[l], wb.k_w[l], wa.k_b[l], wb.k_b[l], 64, s.k));
    PZ_TRY(proj(wa.v_w[l], wb.v_w[l], wa.v_b[l], wb.v_b[l], CATT, s.v));
    prof_mark("attn_qkv_proj", st);
    const int amode = o.attention ? (l == 0 ? 1 : (l == 3 ? 3 : 2)) : 0;
    PZ_TRY(launch_attention(s.q, 64, s.k, 64, s.v, CATT, C, LATT, 64, CATT, x, 1280, s.r, CATT, o.attention, amode, st));
    prof_mark("attn_softmax_av", st);
    GemmF32 g;  // out = x + relu(W_o r + b_o)
    g.A = s.r; g.lda = CATT; g.W[0] = wa.o_w[l]; g.W[1] = wb.o_w[l]; g.bias[0] = wa.o_b[l]; g.bias[1] = wb.o_b[l];
    g.ldw = CATT; g.rows_per_wset = B * LATT; g.Y = att_cat + l * CATT; g.ldy = 1280; g.M = rows; g.N = CATT;
    g.K = CATT; g.relu = 1; g.R = x; g.ldr = 1280;
    PZ_TRY(launch_gemm_f32(g, st));
    prof_mark("attn_out_proj", st);
  }

  // ---- tail: Linear(1280,1024) then max over the 256 points (model5_b.py:472-475)
  GemmF32 g;
  g.A = att_cat; g.lda = 1280; g.W[0] = wa.out_w; g.W[1] = wb.out_w; g.bias[0] = wa.out_b; g.bias[1] = wb.out_b;
  g.ldw = 1280; g.rows_per_wset = B * LATT; g.M = rows; g.N = 1024; g.K = 1280;
  if (o.out) {
    g.Y = o.out; g.ldy = 1024;
    PZ_TRY(launch_gemm_f32(g, st));
    prof_mark("tail_linear", st);
    rowblock_max_kernel<<<dim3(4, C), 256, 0, st>>>(o.out, 1024, LATT, 1024, C, C, 0, c.fglob, 1024);
  } else {
    g.Y = s.tilemax; g.ldy = 1024; g.group = 128;
    PZ_TRY(launch_gemm_f32(g, st));
    prof_mark("tail_linear_maxpool", st);
    rowblock_max_kernel<<<dim3(4, C), 256, 0, st>>>(s.tilemax, 1024, LATT / 128, 1024, C, C, 0, c.fglob, 1024);
  }
  PZ_LAUNCH_CHECK();
  prof_mark("tail_point_max", st);
  return 0;
}

// fglob_pair: optional [B, E*1024] destination laid out for the pose MLP's concat (model5_b.py:723)
static int encoder_forward_impl(const PzEncoderWeights* w, int E, int B, const float* xyz, const int64_t* start1,
                                const int64_t* start2, int precision, const PzEncoderOutputs& o, void* ws,
                                size_t ws_bytes, float* fglob_pair, const AfterStem* after_stem, bool reuse_pack,
                                cudaStream_t st) {
  PZ_REQUIRE(E == 1 || E == 2, PZ_ERR_ARG, "encoder: E must be 1 or 2 (got %d)", E);
  PZ_REQUIRE(B >= 1, PZ_ERR_ARG, "encoder: B must be >= 1");
  PZ_REQUIRE((long long)E * B <= PZ_MAX_CLOUDS, PZ_ERR_UNSUPPORTED, "encoder: E*B = %lld clouds > %d", (long long)E * B,
             PZ_MAX_CLOUDS);
  PZ_REQUIRE(precision == PZ_PREC_FP32 || precision == PZ_PREC_BF16 || precision == PZ_PREC_SPLIT, PZ_ERR_ARG,
             "encoder: unknown precision %d", precision);
  for (int e = 0; e < E; ++e)
    PZ_REQUIRE(encoder_weights_ok(w[e]), PZ_ERR_ARG, "encoder: weight set %d has a null pointer", e);
  const int C = E * B;
  Arena arena(ws, ws_bytes);
  EncoderCommon c;
  Fp32Scratch f = {}; Bf16Scratch b = {}; SplitScratch x = {};
  carve(C, arena, c);
  if (precision == PZ_PREC_FP32) carve(C, arena, f);
  else if (precision == PZ_PREC_BF16) carve(C, arena, b);
  else carve(C, arena, x);
  PZ_REQUIRE(ws && arena.ok(), PZ_ERR_WORKSPACE, "encoder: workspace %zu B < required %zu B", ws_bytes, arena.used);
  if (o.x_feature) c.xfeat = o.x_feature;
  if (o.x2) c.nx2 = o.x2;
  if (o.f_global) c.fglob = o.f_global;

  if (precision == PZ_PREC_FP32) PZ_TRY(encoder_forward_fp32(w, E, B, xyz, start1, start2, o, c, f, after_stem, st));
  else if (precision == PZ_PREC_BF16) PZ_TRY(encoder_forward_bf16(w, E, B, xyz, start1, start2, o, c, b, after_stem, reuse_pack, st));
  else PZ_TRY(encoder_forward_split(w, E, B, xyz, start1, start2, o, c, x, after_stem, reuse_pack, st));

  // f2f = att_cat[:, 1024:1280].  The fp32 path always assembles an fp32 att_cat; without one the tensor-core paths' stage-2
  // GEMM has written f2f directly.
  const float* cat = o.att_cat ? o.att_cat : precision == PZ_PREC_FP32 ? f.att_cat : nullptr;
  if (o.f2f && cat)
    PZ_CUDA(cudaMemcpy2DAsync(o.f2f, CATT * sizeof(float), cat + 4 * CATT, 1280 * sizeof(float), CATT * sizeof(float),
                              (size_t)C * LATT, cudaMemcpyDeviceToDevice, st));
  if (fglob_pair)  // [B, E*1024]: pair b = [f_global(cloud b), f_global(cloud B+b)]
    for (int e = 0; e < E; ++e)
      PZ_CUDA(cudaMemcpy2DAsync(fglob_pair + (size_t)e * 1024, (size_t)E * 1024 * sizeof(float), c.fglob + (size_t)e * B * 1024,
                                1024 * sizeof(float), 1024 * sizeof(float), B, cudaMemcpyDeviceToDevice, st));
  return 0;
}

constexpr size_t HL_SMEM = (3 * 4160 + 64 * 128) * sizeof(float);
constexpr size_t HS_SMEM = (64 * 64 + 32 * 64 + 64 + 32 + 64 + 4 + 64 * 128) * sizeof(float);
static int set_head_fp32_smem() {
  PZ_CUDA(cudaFuncSetAttribute(head_seg_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)HS_SMEM));
  PZ_CUDA(cudaFuncSetAttribute(head_local_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)HL_SMEM));
  return 0;
}

}  // namespace pz

using namespace pz;

// ------------------------------------------------------------------------------ C ABI
extern "C" size_t pz_encoder_workspace_bytes(int E, int B) {
  if (E < 1 || B < 1) return 0;
  auto bytes = [&](auto&& s) {   // the common part, then one precision's layout
    Arena a(nullptr, 0);
    EncoderCommon c;
    carve(E * B, a, c);
    carve(E * B, a, s);
    return a.used;
  };
  return align_up(std::max({bytes(Fp32Scratch()), bytes(Bf16Scratch()), bytes(SplitScratch())}), 256);
}

extern "C" int pz_encoder_forward(const PzEncoderWeights* weights_host, int E, int B, const float* xyz,
                                  const int64_t* start1, const int64_t* start2, int precision,
                                  const PzEncoderOutputs* outputs_host, void* workspace, size_t workspace_bytes,
                                  pz_stream_t stream) {
  PZ_REQUIRE(weights_host && xyz && start1 && start2 && outputs_host, PZ_ERR_ARG, "pz_encoder_forward: null pointer");
  prof_begin(as_stream(stream));
  return encoder_forward_impl(weights_host, E, B, xyz, start1, start2, precision, *outputs_host, workspace,
                              workspace_bytes, nullptr, nullptr, false, as_stream(stream));
}

namespace {
struct PredictScratch {
  float *xyz, *fpair, *h0, *h1, *local, *gmax, *gbias, *tilemax;
  float *x2_all, *attn_all;   // need mode: the encoder's [2B,256,3] / [2B,256,256] outputs, copied out per half
  __nv_bfloat16* himg_split;
  int64_t *st1, *st2;
  void* enc;
  size_t enc_bytes;
};
size_t predict_layout(int B, Arena& a, PredictScratch& s) {
  s.xyz = a.take<float>((size_t)2 * B * NPTS * 3);
  s.st1 = a.take<int64_t>((size_t)2 * B);
  s.st2 = a.take<int64_t>((size_t)2 * B);
  s.fpair = a.take<float>((size_t)B * 2048);
  s.h0 = a.take<float>((size_t)B * 1024);
  s.h1 = a.take<float>((size_t)B * 1024);
  s.local = a.take<float>((size_t)2 * B * NPTS * 64);
  s.gmax = a.take<float>((size_t)B * 64);
  s.gbias = a.take<float>((size_t)2 * B * 64);
  s.tilemax = a.take<float>((size_t)2 * B * 8 * 128);
  s.x2_all = a.take<float>((size_t)2 * B * S2 * 3);
  s.attn_all = a.take<float>((size_t)2 * B * LATT * LATT);
  s.himg_split = a.take<__nv_bfloat16>(2 * HEAD_SPLIT_IMG_SET);
  s.enc_bytes = pz_encoder_workspace_bytes(2, B);
  s.enc = a.take<char>(s.enc_bytes);
  return a.used;
}
}  // namespace

namespace pz {
namespace {
__global__ void __launch_bounds__(256) stage_inputs_kernel(const float4* __restrict__ fpc, const float4* __restrict__ mrpc, size_t n16,
                                                           float4* __restrict__ xyz, const int64_t* __restrict__ starts, int B,
                                                           int64_t* __restrict__ st1, int64_t* __restrict__ st2) {
  pdl_enter();
  const size_t stride = (size_t)gridDim.x * 256;
  for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < 2 * n16; i += stride) xyz[i] = i < n16 ? fpc[i] : mrpc[i - n16];
  if (blockIdx.x == 0) {
    for (int i = threadIdx.x; i < 4 * B; i += 256) {
      const int row = i / B, c = i - row * B;
      ((row & 1) ? st2 : st1)[(row >> 1) * B + c] = starts[i];
    }
  }
}
}  // namespace
}  // namespace pz

extern "C" size_t pz_predict5_workspace_bytes(int B) {
  if (B < 1) return 0;
  Arena a(nullptr, 0);
  PredictScratch s;
  return align_up(predict_layout(B, a, s), 256);
}

namespace {
// pz_predict5's front half, shared with pz_encode_pieces: both clouds into one [2B,1024,3] batch, both encoders, and
// the boundary heads from the encoder's after-stem hook.  local [2B,1024,64] and tilemax [2B,8,64] receive the heads'
// per-cloud state (tilemax on the tensor-core paths only; the fp32 heads pool into s.gmax); the rest of `eo` and
// fglob_pair are as in encoder_forward_impl.
int predict_front(const PzEncoderWeights* enc_host, const PzHeadWeights& h, const float* fpc, const float* mrpc, int B,
                  const int64_t* starts, int precision, bool reuse_pack, const PredictScratch& s,
                  const PzEncoderOutputs& eo, float* fglob_pair, float* local, float* tilemax, float* de_fpcb,
                  float* de_mrpcb, cudaStream_t st) {
  const size_t cloud_bytes = (size_t)B * NPTS * 3 * sizeof(float);
  // both clouds into one [2B, 1024, 3] batch; starts [4,B]: (Encoder s1, Encoder s2, Encoder2 s1, Encoder2 s2) -> st1 =
  // rows 0,2; st2 = rows 1,3.  One launch instead of six copy operations (each ~4 us of stream time).
  if ((((uintptr_t)fpc | (uintptr_t)mrpc) & 15) == 0) {
    PZ_CUDA(launch_pdl(stage_inputs_kernel, dim3(kNumSMs), dim3(256), 0, st, reinterpret_cast<const float4*>(fpc),
                       reinterpret_cast<const float4*>(mrpc), cloud_bytes / 16, reinterpret_cast<float4*>(s.xyz), starts, B, s.st1, s.st2));
    PZ_LAUNCH_CHECK();
  } else {
    PZ_CUDA(cudaMemcpyAsync(s.xyz, fpc, cloud_bytes, cudaMemcpyDeviceToDevice, st));
    PZ_CUDA(cudaMemcpyAsync(s.xyz + (size_t)B * NPTS * 3, mrpc, cloud_bytes, cudaMemcpyDeviceToDevice, st));
    const size_t sb = (size_t)B * sizeof(int64_t);
    PZ_CUDA(cudaMemcpyAsync(s.st1, starts, sb, cudaMemcpyDeviceToDevice, st));
    PZ_CUDA(cudaMemcpyAsync(s.st2, starts + B, sb, cudaMemcpyDeviceToDevice, st));
    PZ_CUDA(cudaMemcpyAsync(s.st1 + B, starts + 2 * (size_t)B, sb, cudaMemcpyDeviceToDevice, st));
    PZ_CUDA(cudaMemcpyAsync(s.st2 + B, starts + 3 * (size_t)B, sb, cudaMemcpyDeviceToDevice, st));
  }

  prof_mark("stage_inputs", st);
  const Mlp3W pre_f = {h.pre_fpc_w[0], h.pre_fpc_b[0], h.pre_fpc_w[1], h.pre_fpc_b[1], h.pre_fpc_w[2], h.pre_fpc_b[2]};
  const Mlp3W pre_r = {h.pre_rpc_w[0], h.pre_rpc_b[0], h.pre_rpc_w[1], h.pre_rpc_b[1], h.pre_rpc_w[2], h.pre_rpc_b[2]};
  const Mlp3W seg_f = {h.seg_fpc_w[0], h.seg_fpc_b[0], h.seg_fpc_w[1], h.seg_fpc_b[1], h.seg_fpc_w[2], h.seg_fpc_b[2]};
  const Mlp3W seg_r = {h.seg_rpc_w[0], h.seg_rpc_b[0], h.seg_rpc_w[1], h.seg_rpc_b[1], h.seg_rpc_w[2], h.seg_rpc_b[2]};
  const int P = 2 * B * NPTS;

  // boundary heads (model5_b.py:738-754): they only need x_feature, so the encoder runs them right after its stem
  AfterStem heads_fn = [&](const float* xfeat) -> int {
    if (precision == PZ_PREC_SPLIT || precision == PZ_PREC_BF16) {
      // split-fp16 chained-MMA heads on the fp32 x_feature (heads_split.cu): logits at fp32 tolerance in both
      // tensor-core precisions (the bf16 path's stem is a split product too, so its x_feature is fp32-accurate)
      PZ_TRY(launch_heads_split(xfeat, pre_f, pre_r, seg_f, seg_r, B, reuse_pack, s.himg_split, local, tilemax, de_fpcb,
                                de_mrpcb, st));
      prof_mark("boundary_heads", st);
      return 0;
    }
    PZ_TRY(set_head_fp32_smem());
    head_local_kernel<<<P / 128, 128, HL_SMEM, st>>>(xfeat, pre_f, pre_r, B, local);
    PZ_LAUNCH_CHECK();
    // D6: BOTH heads use the max-pool of the *mrpc* local features (model5_b.py:741-744)
    rowblock_max_kernel<<<dim3(1, B), 256, 0, st>>>(local + (size_t)B * NPTS * 64, 64, NPTS, 64, B, B, 0, s.gmax, 64);
    PZ_LAUNCH_CHECK();
    seg_bias_kernel<<<dim3(B, 2), 64, 0, st>>>(s.gmax, 1, nullptr, h.seg_fpc_w[0], h.seg_fpc_b[0], h.seg_rpc_w[0],
                                               h.seg_rpc_b[0], B, s.gbias);
    PZ_LAUNCH_CHECK();
    head_seg_kernel<<<P / 128, 128, HS_SMEM, st>>>(local, seg_f, seg_r, s.gbias, B, de_fpcb, de_mrpcb, nullptr);
    PZ_LAUNCH_CHECK();
    prof_mark("boundary_heads", st);
    return 0;
  };

  return encoder_forward_impl(enc_host, 2, B, s.xyz, s.st1, s.st2, precision, eo, s.enc, s.enc_bytes, fglob_pair,
                              &heads_fn, reuse_pack, st);
}

// null-pointer check of every head weight
int check_heads(const PzHeadWeights* heads_host, const char* who) {
  const void* const* p = reinterpret_cast<const void* const*>(heads_host);
  for (size_t i = 0; i < sizeof(PzHeadWeights) / sizeof(void*); ++i)
    PZ_REQUIRE(p[i], PZ_ERR_ARG, "%s: head weight %zu is null", who, i);
  return 0;
}

// pose MLP on rows of cat(ffpc, fmrpc) (model5_b.py:723-725): 2048-1024-512-512-256-6, fp32 in every precision
int pose_mlp(const PzHeadWeights& h, const float* fpair, int n, float* h0, float* h1, float* out6, cudaStream_t st) {
  PZ_TRY(skinny_linear(fpair, 2048, h.tf_w[0], h.tf_b[0], n, 1024, 2048, 1, h0, 1024, st));
  PZ_TRY(skinny_linear(h0, 1024, h.tf_w[1], h.tf_b[1], n, 512, 1024, 1, h1, 512, st));
  PZ_TRY(skinny_linear(h1, 512, h.tf_w[2], h.tf_b[2], n, 512, 512, 1, h0, 512, st));
  PZ_TRY(skinny_linear(h0, 512, h.tf_w[3], h.tf_b[3], n, 256, 512, 1, h1, 256, st));
  PZ_TRY(skinny_linear(h1, 256, h.tf_w[4], h.tf_b[4], n, 6, 256, 0, out6, 6, st));
  prof_mark("pose_mlp", st);
  return 0;
}
}  // namespace

extern "C" int pz_predict5(const PzEncoderWeights* enc_host, const PzHeadWeights* heads_host, const float* fpc,
                           const float* mrpc, int B, const int64_t* starts, int precision, int flags, float* out6,
                           float* de_fpcb, float* de_mrpcb, float* x2_fpc, float* attention_fpc, float* x2_mrpc,
                           float* attention_mrpc, void* workspace, size_t workspace_bytes, pz_stream_t stream) {
  PZ_REQUIRE(enc_host && heads_host && fpc && mrpc && starts && out6 && de_fpcb && de_mrpcb, PZ_ERR_ARG,
             "pz_predict5: null pointer");
  PZ_REQUIRE(B >= 1, PZ_ERR_ARG, "pz_predict5: B must be >= 1");
  PZ_REQUIRE(B <= PZ_MAX_CLOUDS / 2, PZ_ERR_UNSUPPORTED, "pz_predict5: B = %d > %d (2B clouds)", B, PZ_MAX_CLOUDS / 2);
  const int need = flags & PZ_FLAG_NEED;
  const bool reuse_pack = (flags & PZ_FLAG_REUSE_PACKS) != 0;
  if (need)
    PZ_REQUIRE(x2_fpc && attention_fpc && x2_mrpc && attention_mrpc, PZ_ERR_ARG,
               "pz_predict5: need=1 requires the x2/attention outputs");
  PZ_TRY(check_heads(heads_host, "pz_predict5"));
  cudaStream_t st = as_stream(stream);
  Arena arena(workspace, workspace_bytes);
  PredictScratch s;
  predict_layout(B, arena, s);
  PZ_REQUIRE(workspace && arena.ok(), PZ_ERR_WORKSPACE, "pz_predict5: workspace %zu B < required %zu B",
             workspace_bytes, arena.used);
  prof_begin(st);
  PzEncoderOutputs eo = {};
  if (need) {   // the encoder writes contiguous [2B,..] tensors; the caller's four outputs are separate
    eo.attention = s.attn_all;
    eo.x2 = s.x2_all;
  }
  const PzHeadWeights& h = *heads_host;
  PZ_TRY(predict_front(enc_host, h, fpc, mrpc, B, starts, precision, reuse_pack, s, eo, s.fpair, s.local, s.tilemax,
                       de_fpcb, de_mrpcb, st));
  if (need) {
    const size_t ab = (size_t)B * LATT * LATT * sizeof(float), xb = (size_t)B * S2 * 3 * sizeof(float);
    PZ_CUDA(cudaMemcpyAsync(attention_fpc, s.attn_all, ab, cudaMemcpyDeviceToDevice, st));
    PZ_CUDA(cudaMemcpyAsync(attention_mrpc, s.attn_all + (size_t)B * LATT * LATT, ab, cudaMemcpyDeviceToDevice, st));
    PZ_CUDA(cudaMemcpyAsync(x2_fpc, s.x2_all, xb, cudaMemcpyDeviceToDevice, st));
    PZ_CUDA(cudaMemcpyAsync(x2_mrpc, s.x2_all + (size_t)B * S2 * 3, xb, cudaMemcpyDeviceToDevice, st));
  }
  return pose_mlp(h, s.fpair, B, s.h0, s.h1, out6, st);
}

// ------------------------------------------------------------- pair scoring from per-piece encodings
namespace {
size_t encode_layout(int P, Arena& a, PredictScratch& s, float** de_fpcb_diag) {
  predict_layout(P, a, s);
  *de_fpcb_diag = a.take<float>((size_t)P * 2 * NPTS);   // the fpc head of the diagonal pairs: computed, not kept
  return a.used;
}
// every embedding buffer is read or written with 16-byte vector accesses
bool embeddings_aligned(const PzPieceEmbeddings& e) {
  return ((((uintptr_t)e.f_global | (uintptr_t)e.local | (uintptr_t)e.tilemax | (uintptr_t)e.de_mrpcb)) & 15) == 0;
}
struct PairScratch {
  float *fpair, *h0, *h1, *gbias;
  __half* himg_split;
};
size_t pairs_layout(int n, Arena& a, PairScratch& s) {
  s.himg_split = a.take<__half>(2 * HEAD_SPLIT_IMG_SET);   // first: its offset does not depend on n
  s.fpair = a.take<float>((size_t)n * 2048);
  s.h0 = a.take<float>((size_t)n * 1024);
  s.h1 = a.take<float>((size_t)n * 1024);
  s.gbias = a.take<float>((size_t)n * 64);
  return a.used;
}
}  // namespace

namespace pz {
namespace {
// per pair p = (i, j): fpair[p] = [f_global[0,i], f_global[1,j]] (the pose MLP's input row) and de_out[p] = de_mrpcb[j]
__global__ void __launch_bounds__(256) gather_pair_rows_kernel(const float4* __restrict__ fg, int P,
                                                               const float4* __restrict__ de_mrpcb,
                                                               const int64_t* __restrict__ pairs,
                                                               float4* __restrict__ fpair, float4* __restrict__ de_out) {
  pdl_enter();
  const int p = blockIdx.x, t = threadIdx.x;   // 256 threads x 2 float4 = one 2048-float row of each output
  const size_t i = (size_t)pairs[2 * p], j = (size_t)pairs[2 * p + 1];
  fpair[(size_t)p * 512 + t] = fg[i * 256 + t];
  fpair[(size_t)p * 512 + 256 + t] = fg[((size_t)P + j) * 256 + t];
  de_out[(size_t)p * 512 + t] = de_mrpcb[j * 512 + t];
  de_out[(size_t)p * 512 + 256 + t] = de_mrpcb[j * 512 + 256 + t];
}
}  // namespace
}  // namespace pz

extern "C" size_t pz_encode_pieces_workspace_bytes(int P) {
  if (P < 1) return 0;
  Arena a(nullptr, 0);
  PredictScratch s;
  float* de;
  return align_up(encode_layout(P, a, s, &de), 256);
}

extern "C" int pz_encode_pieces(const PzEncoderWeights* enc_host, const PzHeadWeights* heads_host, const float* clouds,
                                int P, const int64_t* starts, int precision, int flags, const PzPieceEmbeddings* emb_host,
                                void* workspace, size_t workspace_bytes, pz_stream_t stream) {
  PZ_REQUIRE(enc_host && heads_host && clouds && starts && emb_host, PZ_ERR_ARG, "pz_encode_pieces: null pointer");
  const PzPieceEmbeddings& e = *emb_host;
  PZ_REQUIRE(e.f_global && e.local && e.tilemax && e.de_mrpcb, PZ_ERR_ARG, "pz_encode_pieces: null embedding pointer");
  PZ_REQUIRE(P >= 1, PZ_ERR_ARG, "pz_encode_pieces: P must be >= 1");
  PZ_REQUIRE(P <= PZ_MAX_PIECES, PZ_ERR_UNSUPPORTED, "pz_encode_pieces: P = %d > %d", P, PZ_MAX_PIECES);
  PZ_REQUIRE(embeddings_aligned(e), PZ_ERR_ARG, "pz_encode_pieces: embedding buffers must be 16-byte aligned");
  PZ_REQUIRE(precision == PZ_PREC_FP32 || precision == PZ_PREC_BF16 || precision == PZ_PREC_SPLIT, PZ_ERR_ARG,
             "pz_encode_pieces: unknown precision %d", precision);
  PZ_REQUIRE(!(flags & PZ_FLAG_NEED), PZ_ERR_UNSUPPORTED, "pz_encode_pieces: PZ_FLAG_NEED is not supported");
  PZ_TRY(check_heads(heads_host, "pz_encode_pieces"));
  cudaStream_t st = as_stream(stream);
  Arena arena(workspace, workspace_bytes);
  PredictScratch s;
  float* de_fpcb_diag = nullptr;
  encode_layout(P, arena, s, &de_fpcb_diag);
  PZ_REQUIRE(workspace && arena.ok(), PZ_ERR_WORKSPACE, "pz_encode_pieces: workspace %zu B < required %zu B",
             workspace_bytes, arena.used);
  prof_begin(st);
  PzEncoderOutputs eo = {};
  eo.f_global = e.f_global;   // [2P,1024] == [2,P,1024]: cloud c < P is piece c through Encoder, c >= P through Encoder2
  PZ_TRY(predict_front(enc_host, *heads_host, clouds, clouds, P, starts, precision, (flags & PZ_FLAG_REUSE_PACKS) != 0,
                       s, eo, nullptr, e.local, e.tilemax, de_fpcb_diag, e.de_mrpcb, st));
  if (precision == PZ_PREC_FP32) {   // the fp32 heads pool whole clouds; the embeddings keep the per-tile maxima
    rowblock_max_kernel<<<dim3(1, 2 * P * 8), 256, 0, st>>>(e.local, 64, 128, 64, 2 * P * 8, 2 * P * 8, 0, e.tilemax, 64);
    PZ_LAUNCH_CHECK();
  }
  return 0;
}

extern "C" size_t pz_predict_pairs_workspace_bytes(int n) {
  if (n < 1) return 0;
  Arena a(nullptr, 0);
  PairScratch s;
  return align_up(pairs_layout(n, a, s), 256);
}

extern "C" int pz_predict_pairs(const PzHeadWeights* heads_host, const PzPieceEmbeddings* emb_host, int P,
                                const int64_t* pairs, int n, int precision, int flags, float* out6, float* de_fpcb,
                                float* de_mrpcb, void* workspace, size_t workspace_bytes, pz_stream_t stream) {
  PZ_REQUIRE(n >= 0, PZ_ERR_ARG, "pz_predict_pairs: n < 0");
  if (n == 0) return 0;
  PZ_REQUIRE(heads_host && emb_host && pairs && out6 && de_fpcb && de_mrpcb, PZ_ERR_ARG, "pz_predict_pairs: null pointer");
  const PzPieceEmbeddings& e = *emb_host;
  PZ_REQUIRE(e.f_global && e.local && e.tilemax && e.de_mrpcb, PZ_ERR_ARG, "pz_predict_pairs: null embedding pointer");
  PZ_REQUIRE(P >= 1, PZ_ERR_ARG, "pz_predict_pairs: P must be >= 1");
  PZ_REQUIRE(n <= PZ_MAX_PAIRS, PZ_ERR_UNSUPPORTED, "pz_predict_pairs: n = %d > %d", n, PZ_MAX_PAIRS);
  PZ_REQUIRE(precision == PZ_PREC_FP32 || precision == PZ_PREC_BF16 || precision == PZ_PREC_SPLIT, PZ_ERR_ARG,
             "pz_predict_pairs: unknown precision %d", precision);
  PZ_REQUIRE(!(flags & PZ_FLAG_NEED), PZ_ERR_UNSUPPORTED, "pz_predict_pairs: PZ_FLAG_NEED is not supported");
  PZ_TRY(check_heads(heads_host, "pz_predict_pairs"));
  PZ_REQUIRE(embeddings_aligned(e) && ((uintptr_t)de_mrpcb & 15) == 0, PZ_ERR_ARG,
             "pz_predict_pairs: embedding buffers and de_mrpcb must be 16-byte aligned");
  cudaStream_t st = as_stream(stream);
  Arena arena(workspace, workspace_bytes);
  PairScratch s;
  pairs_layout(n, arena, s);
  PZ_REQUIRE(workspace && arena.ok(), PZ_ERR_WORKSPACE, "pz_predict_pairs: workspace %zu B < required %zu B",
             workspace_bytes, arena.used);
  prof_begin(st);
  const PzHeadWeights& h = *heads_host;
  const Mlp3W pre_f = {h.pre_fpc_w[0], h.pre_fpc_b[0], h.pre_fpc_w[1], h.pre_fpc_b[1], h.pre_fpc_w[2], h.pre_fpc_b[2]};
  const Mlp3W pre_r = {h.pre_rpc_w[0], h.pre_rpc_b[0], h.pre_rpc_w[1], h.pre_rpc_b[1], h.pre_rpc_w[2], h.pre_rpc_b[2]};
  const Mlp3W seg_f = {h.seg_fpc_w[0], h.seg_fpc_b[0], h.seg_fpc_w[1], h.seg_fpc_b[1], h.seg_fpc_w[2], h.seg_fpc_b[2]};
  const Mlp3W seg_r = {h.seg_rpc_w[0], h.seg_rpc_b[0], h.seg_rpc_w[1], h.seg_rpc_b[1], h.seg_rpc_w[2], h.seg_rpc_b[2]};
  const float* tilemax_mrpc = e.tilemax + (size_t)P * 8 * 64;
  PZ_CUDA(launch_pdl(gather_pair_rows_kernel, dim3(n), dim3(256), 0, st, reinterpret_cast<const float4*>(e.f_global), P,
                     reinterpret_cast<const float4*>(e.de_mrpcb), pairs, reinterpret_cast<float4*>(s.fpair),
                     reinterpret_cast<float4*>(de_mrpcb)));
  PZ_LAUNCH_CHECK();
  prof_mark("gather_pairs", st);
  if (precision == PZ_PREC_FP32) {
    PZ_TRY(set_head_fp32_smem());
    seg_bias_kernel<<<dim3(n, 1), 64, 0, st>>>(tilemax_mrpc, 8, pairs, h.seg_fpc_w[0], h.seg_fpc_b[0], h.seg_rpc_w[0],
                                               h.seg_rpc_b[0], n, s.gbias);
    PZ_LAUNCH_CHECK();
    head_seg_kernel<<<n * NPTS / 128, 128, HS_SMEM, st>>>(e.local, seg_f, seg_r, s.gbias, n, de_fpcb, nullptr, pairs);
    PZ_LAUNCH_CHECK();
  } else {
    PZ_TRY(launch_seg_pairs_split(pre_f, pre_r, seg_f, seg_r, (flags & PZ_FLAG_REUSE_PACKS) != 0, s.himg_split, e.local,
                                  tilemax_mrpc, pairs, n, de_fpcb, st));
  }
  prof_mark("boundary_heads", st);
  return pose_mlp(h, s.fpair, n, s.h0, s.h1, out6, st);
}

extern "C" int pz_se3_exp(const float* twist, int B, float* g, pz_stream_t stream) {
  PZ_REQUIRE(twist && g, PZ_ERR_ARG, "pz_se3_exp: null pointer");
  PZ_REQUIRE(B >= 0, PZ_ERR_ARG, "pz_se3_exp: B < 0");
  if (B == 0) return 0;
  se3_exp_kernel<<<(B + 127) / 128, 128, 0, as_stream(stream)>>>(twist, B, g);
  PZ_LAUNCH_CHECK();
  return 0;
}

extern "C" int pz_scaled_dot_attention(const float* q, const float* k, const float* v, int B, int L, int Dk, int Dv,
                                       float* values, float* attention_or_null, pz_stream_t stream) {
  PZ_REQUIRE(q && k && v && values, PZ_ERR_ARG, "pz_scaled_dot_attention: null pointer");
  PZ_REQUIRE(B >= 0, PZ_ERR_ARG, "pz_scaled_dot_attention: B < 0");
  if (B == 0) return 0;
  return launch_attention(q, Dk, k, Dk, v, Dv, B, L, Dk, Dv, nullptr, 0, values, Dv, attention_or_null,
                          attention_or_null ? 1 : 0, as_stream(stream));
}

extern "C" int pz_linear(const float* x, int ldx, const float* W, const float* b, int M, int N, int K, int relu,
                         const float* residual_or_null, int ldr, float* y, int ldy, int precision,
                         pz_stream_t stream) {
  PZ_REQUIRE(x && W && y, PZ_ERR_ARG, "pz_linear: null pointer");
  PZ_REQUIRE(M >= 0 && N >= 1 && K >= 1 && ldx >= K && ldy >= N, PZ_ERR_ARG, "pz_linear: bad sizes");
  PZ_REQUIRE(precision == PZ_PREC_FP32, PZ_ERR_UNSUPPORTED, "pz_linear: precision %d not available", precision);
  if (M == 0) return 0;
  GemmF32 g;
  g.A = x; g.lda = ldx; g.W[0] = W; g.bias[0] = b; g.ldw = K; g.Y = y; g.ldy = ldy; g.M = M; g.N = N; g.K = K;
  g.relu = relu; g.R = residual_or_null; g.ldr = ldr;
  return launch_gemm_f32(g, as_stream(stream));
}

namespace {
// pz_offset_attention's workspace: one layout per precision over rows = B * L rows of C channels
struct OffsetAttnFp32 { float *q, *k, *v, *r; };
size_t layout(Arena& a, size_t rows, int C, OffsetAttnFp32& s) {
  s.q = a.take<float>(rows * (C / 4));
  s.k = a.take<float>(rows * (C / 4));
  s.v = a.take<float>(rows * C);
  s.r = a.take<float>(rows * C);
  return a.used;
}
// bf16: x and out, one layer's weight tile images, the q|k|v bias
struct OffsetAttnBf16 { __nv_bfloat16 *x, *y, *wimg; float* bqkv; };
size_t layout(Arena& a, size_t rows, int C, OffsetAttnBf16& s) {
  s.x = a.take<__nv_bfloat16>(rows * C);
  s.y = a.take<__nv_bfloat16>(rows * C);
  s.wimg = a.take<__nv_bfloat16>(ATTN_WIMG_ELEMS);
  s.bqkv = a.take<float>(384);
  return a.used;
}
// split, [plane]: x, q|k, v^T, r, the four weights (rows: q 0-63, k 64-127, v 128-383, o 384-639), the q|k|v bias
struct OffsetAttnSplit { h16 *x[2], *qk[2], *vT[2], *r[2], *w[2]; float* bqkv; };
size_t layout(Arena& a, size_t rows, int C, OffsetAttnSplit& s) {
  s.x[0] = a.take<h16>(rows * C); s.x[1] = a.take<h16>(rows * C);
  s.qk[0] = a.take<h16>(rows * 128); s.qk[1] = a.take<h16>(rows * 128);
  s.vT[0] = a.take<h16>(rows * C); s.vT[1] = a.take<h16>(rows * C);
  s.r[0] = a.take<h16>(rows * C); s.r[1] = a.take<h16>(rows * C);
  s.w[0] = a.take<h16>((size_t)640 * C); s.w[1] = a.take<h16>((size_t)640 * C);
  s.bqkv = a.take<float>(384);
  return a.used;
}
}  // namespace

extern "C" size_t pz_offset_attention_workspace_bytes(int B, int L, int C) {
  if (B < 1 || L < 1 || C < 4) return 0;
  auto bytes = [&](auto&& s) {
    Arena a(nullptr, 0);
    return layout(a, (size_t)B * L, C, s);
  };
  return align_up(std::max({bytes(OffsetAttnFp32()), bytes(OffsetAttnBf16()), bytes(OffsetAttnSplit())}), 256);
}

extern "C" int pz_offset_attention(const float* x, const float* Wq, const float* bq, const float* Wk, const float* bk,
                                   const float* Wv, const float* bv, const float* Wo, const float* bo, int B, int L,
                                   int C, int precision, float* out, float* attention_or_null, void* workspace,
                                   size_t workspace_bytes, pz_stream_t stream) {
  PZ_REQUIRE(x && Wq && bq && Wk && bk && Wv && bv && Wo && bo && out, PZ_ERR_ARG, "pz_offset_attention: null pointer");
  PZ_REQUIRE(B >= 1 && C == 256, PZ_ERR_UNSUPPORTED, "pz_offset_attention: C must be 256 (got %d)", C);
  PZ_REQUIRE(precision == PZ_PREC_FP32 || precision == PZ_PREC_BF16 || precision == PZ_PREC_SPLIT, PZ_ERR_ARG,
             "pz_offset_attention: unknown precision %d", precision);
  cudaStream_t st = as_stream(stream);
  Arena a(workspace, workspace_bytes);
  PZ_REQUIRE(precision == PZ_PREC_FP32 || L == 256, PZ_ERR_UNSUPPORTED, "pz_offset_attention(%s): L must be 256 (got %d)",
             precision == PZ_PREC_SPLIT ? "split" : "bf16", L);
  const size_t rows = (size_t)B * L;
  OffsetAttnFp32 f = {}; OffsetAttnBf16 b = {}; OffsetAttnSplit s = {};
  if (precision == PZ_PREC_SPLIT) layout(a, rows, C, s);
  else if (precision == PZ_PREC_BF16) layout(a, rows, C, b);
  else layout(a, rows, C, f);
  PZ_REQUIRE(workspace && a.ok(), PZ_ERR_WORKSPACE, "pz_offset_attention: workspace %zu B < required %zu B",
             workspace_bytes, a.used);
  if (precision == PZ_PREC_SPLIT) {   // the split path's layer: row GEMMs + attention_split_kernel (gemm_split.cu, attention_split.cu)
    PackJobs jobs;
    int n = 0;
    for (int pl = 0; pl < 2; ++pl) {
      h16* w = s.w[pl];
      jobs.j[n++] = PackJob{Wq, w, C, 64, C, C, 4 + pl};
      jobs.j[n++] = PackJob{Wk, w + 64 * C, C, 64, C, C, 4 + pl};
      jobs.j[n++] = PackJob{Wv, w + 128 * C, C, C, C, C, 4 + pl};
      jobs.j[n++] = PackJob{Wo, w + 384 * C, C, C, C, C, 4 + pl};
    }
    jobs.j[n++] = PackJob{bq, s.bqkv, 64, 1, 64, 64, 0};
    jobs.j[n++] = PackJob{bk, s.bqkv + 64, 64, 1, 64, 64, 0};
    jobs.j[n++] = PackJob{bv, s.bqkv + 128, C, 1, C, C, 0};
    jobs.n = n;
    pack_weights_kernel<<<dim3(16, n), 256, 0, st>>>(jobs);
    PZ_LAUNCH_CHECK();
    PZ_TRY(launch_split_planes(x, C, rows, C, s.x[0], s.x[1], C, st));
    TcGemm gq;
    gq.X = s.x[0]; gq.Xlo = s.x[1]; gq.ldx = C; gq.W[0] = s.w[0]; gq.Wlo[0] = s.w[1]; gq.ldw = C; gq.bias[0] = s.bqkv;
    gq.M = (int)rows; gq.Nout = 128; gq.K = C; gq.Yb = s.qk[0]; gq.Yblo = s.qk[1]; gq.ldyb = 128;
    PZ_TRY(launch_split_rowgemm(gq, st));
    TcGemm gv = gq;
    gv.W[0] = s.w[0] + 128 * C; gv.Wlo[0] = s.w[1] + 128 * C; gv.bias[0] = s.bqkv + 128; gv.Nout = C; gv.Yb = nullptr; gv.Yblo = nullptr;
    gv.YT = s.vT[0]; gv.YTlo = s.vT[1]; gv.t_rows = L;
    PZ_TRY(launch_split_rowgemm(gv, st));
    AttnSplit ap;
    ap.qk_hi = s.qk[0]; ap.qk_lo = s.qk[1]; ap.vT_hi = s.vT[0]; ap.vT_lo = s.vT[1]; ap.x_hi = s.x[0]; ap.x_lo = s.x[1]; ap.ldx = C;
    ap.r_hi = s.r[0]; ap.r_lo = s.r[1];
    ap.attn = attention_or_null; ap.attn_mode = attention_or_null ? 1 : 0;
    PZ_TRY(launch_attention_split(ap, B, st));
    TcGemm go;
    go.X = s.r[0]; go.Xlo = s.r[1]; go.ldx = C; go.W[0] = s.w[0] + 384 * C; go.Wlo[0] = s.w[1] + 384 * C; go.ldw = C; go.bias[0] = bo;
    go.M = (int)rows; go.Nout = C; go.K = C; go.relu = 1; go.Rf = x; go.ldrf = C; go.Yf = out; go.ldyf = C;
    return launch_split_rowgemm(go, st);
  }
  if (precision == PZ_PREC_BF16) {   // the fused tcgen05 layer kernel predict5 uses (attention_layer_tc.cu)
    PZ_TRY(launch_cvt_bf16(x, C, (int)rows, C, b.x, C, st));
    PZ_TRY(launch_attn_weight_image(Wq, 64, 0, b.wimg, st));
    PZ_TRY(launch_attn_weight_image(Wk, 64, 64, b.wimg, st));
    PZ_TRY(launch_attn_weight_image(Wv, C, 128, b.wimg, st));
    PZ_TRY(launch_attn_weight_image(Wo, C, 384, b.wimg, st));
    PZ_CUDA(cudaMemcpyAsync(b.bqkv, bq, 64 * sizeof(float), cudaMemcpyDeviceToDevice, st));
    PZ_CUDA(cudaMemcpyAsync(b.bqkv + 64, bk, 64 * sizeof(float), cudaMemcpyDeviceToDevice, st));
    PZ_CUDA(cudaMemcpyAsync(b.bqkv + 128, bv, C * sizeof(float), cudaMemcpyDeviceToDevice, st));
    AttnLayerTc p;
    p.nlayers = 1;
    p.x = b.x; p.ldx = C; p.wimg[0] = p.wimg[1] = b.wimg; p.bqkv[0] = p.bqkv[1] = b.bqkv; p.bo[0][0] = p.bo[1][0] = bo;
    p.clouds_per_set = B; p.yb = b.y; p.ldyb = C; p.yf = out; p.ldyf = C;
    p.attn = attention_or_null; p.attn_mode[0] = attention_or_null ? 1 : 0;
    return launch_attention_layer_tc(p, B, st);
  }
  auto lin = [&](const float* in, const float* W, const float* b, int N, float* y, int relu, const float* R) {
    GemmF32 g;
    g.A = in; g.lda = C; g.W[0] = W; g.bias[0] = b; g.ldw = C; g.Y = y; g.ldy = N; g.M = (int)rows; g.N = N; g.K = C;
    g.relu = relu; g.R = R; g.ldr = C;
    return launch_gemm_f32(g, st);
  };
  PZ_TRY(lin(x, Wq, bq, C / 4, f.q, 0, nullptr));
  PZ_TRY(lin(x, Wk, bk, C / 4, f.k, 0, nullptr));
  PZ_TRY(lin(x, Wv, bv, C, f.v, 0, nullptr));
  PZ_TRY(launch_attention(f.q, C / 4, f.k, C / 4, f.v, C, B, L, C / 4, C, x, C, f.r, C, attention_or_null,
                          attention_or_null ? 1 : 0, st));
  return lin(f.r, Wo, bo, C, out, 1, x);
}

namespace {
// pz_group_mlp_maxpool's workspace: the int32 neighbour rows [B*S*K], then one layout per precision (pts = B * N source
// points, centres = B * S)
struct GroupMlpFp32 { float* F; };   // the feature half of layer 1 [pts, C1]
size_t layout(Arena& a, size_t pts, size_t, int, int C1, int, GroupMlpFp32& s) {
  s.F = a.take<float>(pts * C1);
  return a.used;
}
struct GroupMlpBf16 { __nv_bfloat16 *feat, *P, *w1f, *w2; };   // feat [pts, D], P [pts, C1], W1[:,3:] [C1, D], W2 [C2, C1]
size_t layout(Arena& a, size_t pts, size_t, int D, int C1, int C2, GroupMlpBf16& s) {
  s.feat = a.take<__nv_bfloat16>(pts * D);
  s.P = a.take<__nv_bfloat16>(pts * C1);
  s.w1f = a.take<__nv_bfloat16>((size_t)C1 * D);
  s.w2 = a.take<__nv_bfloat16>((size_t)C2 * C1);
  return a.used;
}
struct GroupMlpSplit { h16 *feat[2], *w1f[2], *w2[2]; float *P, *Q; };   // [plane]; P [pts, C1], Q [centres, C1]
size_t layout(Arena& a, size_t pts, size_t centres, int D, int C1, int C2, GroupMlpSplit& s) {
  s.feat[0] = a.take<h16>(pts * D); s.feat[1] = a.take<h16>(pts * D);
  s.P = a.take<float>(pts * C1);
  s.Q = a.take<float>(centres * C1);
  s.w1f[0] = a.take<h16>((size_t)C1 * D); s.w1f[1] = a.take<h16>((size_t)C1 * D);
  s.w2[0] = a.take<h16>((size_t)C2 * C1); s.w2[1] = a.take<h16>((size_t)C2 * C1);
  return a.used;
}
}  // namespace

extern "C" size_t pz_group_mlp_workspace_bytes(int B, int N, int D, int S, int K, int C1, int C2) {
  if (B < 1 || N < 1 || S < 1 || K < 1 || C1 < 1 || C2 < 1 || D < 1) return 0;
  auto bytes = [&](auto&& s) {
    Arena a(nullptr, 0);
    a.take<int>((size_t)B * S * K);
    return layout(a, (size_t)B * N, (size_t)B * S, D, C1, C2, s);
  };
  return align_up(std::max({bytes(GroupMlpFp32()), bytes(GroupMlpBf16()), bytes(GroupMlpSplit())}), 256);
}

extern "C" int pz_group_mlp_maxpool(const float* xyz, const float* feat, const float* new_xyz, const int64_t* knn_idx,
                                    const float* W1, const float* b1, const float* W2, const float* b2, int B, int N,
                                    int D, int S, int K, int C1, int C2, int precision, float* out, void* workspace,
                                    size_t workspace_bytes, pz_stream_t stream) {
  PZ_REQUIRE(xyz && feat && new_xyz && knn_idx && W1 && b1 && W2 && b2 && out, PZ_ERR_ARG,
             "pz_group_mlp_maxpool: null pointer");
  PZ_REQUIRE(B >= 1 && N >= 1 && D >= 1 && S >= 1 && C1 >= 1 && C2 >= 1, PZ_ERR_ARG, "pz_group_mlp_maxpool: bad sizes");
  PZ_REQUIRE(K == 32, PZ_ERR_UNSUPPORTED, "pz_group_mlp_maxpool: K must be 32 (got %d)", K);
  PZ_REQUIRE(C1 <= 256, PZ_ERR_UNSUPPORTED, "pz_group_mlp_maxpool: C1 must be <= 256 (got %d)", C1);
  PZ_REQUIRE(((size_t)B * S * K) % 128 == 0, PZ_ERR_UNSUPPORTED, "pz_group_mlp_maxpool: B*S must be a multiple of 4");
  // grouped rows (GEMM M) and source-point row ids (B*N) are 32-bit ints on the device
  PZ_REQUIRE((size_t)B * S * K <= INT_MAX && (size_t)B * N <= INT_MAX, PZ_ERR_UNSUPPORTED,
             "pz_group_mlp_maxpool: B*S*K = %zu and B*N = %zu must not exceed %d", (size_t)B * S * K, (size_t)B * N,
             INT_MAX);
  PZ_REQUIRE(precision == PZ_PREC_FP32 || precision == PZ_PREC_BF16 || precision == PZ_PREC_SPLIT, PZ_ERR_ARG,
             "pz_group_mlp_maxpool: unknown precision %d", precision);
  PZ_REQUIRE(precision == PZ_PREC_FP32 || (D % 64 == 0 && (C1 == 128 || C1 == 256) && (C2 == 128 || C2 == 256) &&
                                             ((size_t)B * N) % 128 == 0 && ((size_t)B * S * K) % 256 == 0),
             PZ_ERR_UNSUPPORTED,
             "pz_group_mlp_maxpool(%s): needs D %% 64 == 0, C1,C2 in {128,256}, B*N %% 128 == 0, B*S %% 8 == 0",
             precision == PZ_PREC_SPLIT ? "split" : "bf16");
  cudaStream_t st = as_stream(stream);
  Arena a(workspace, workspace_bytes);
  const size_t total = (size_t)B * S * K, pts = (size_t)B * N, centres = (size_t)B * S;
  int* rows = a.take<int>(total);
  GroupMlpFp32 f = {}; GroupMlpBf16 b = {}; GroupMlpSplit s = {};
  if (precision == PZ_PREC_SPLIT) layout(a, pts, centres, D, C1, C2, s);
  else if (precision == PZ_PREC_BF16) layout(a, pts, centres, D, C1, C2, b);
  else layout(a, pts, centres, D, C1, C2, f);
  PZ_REQUIRE(workspace && a.ok(), PZ_ERR_WORKSPACE, "pz_group_mlp_maxpool: workspace %zu B < required %zu B",
             workspace_bytes, a.used);
  idx64_to_rows32_kernel<<<(int)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096), 256, 0, st>>>(
      knn_idx, total, (size_t)S * K, N, rows);
  PZ_LAUNCH_CHECK();
  if (precision == PZ_PREC_SPLIT) {
    // split path: P = feat W1[:,3:]^T + b1 + W1[:,0:3] xyz and Q = W1[:,0:3] c in fp32, then the split gather GEMM
    PackJobs jobs;
    jobs.j[0] = PackJob{W1 + 3, s.w1f[0], 3 + D, C1, D, D, 4};
    jobs.j[1] = PackJob{W1 + 3, s.w1f[1], 3 + D, C1, D, D, 5};
    jobs.j[2] = PackJob{W2, s.w2[0], C1, C2, C1, C1, 4};
    jobs.j[3] = PackJob{W2, s.w2[1], C1, C2, C1, C1, 5};
    jobs.n = 4;
    pack_weights_kernel<<<dim3(16, 4), 256, 0, st>>>(jobs);
    PZ_LAUNCH_CHECK();
    PZ_TRY(launch_split_planes(feat, D, pts, D, s.feat[0], s.feat[1], D, st));
    PZ_TRY(launch_centre_proj_f32(new_xyz, W1, W1, 3 + D, B * S, B * S, C1, s.Q, st));
    TcGemm g1;
    g1.X = s.feat[0]; g1.Xlo = s.feat[1]; g1.ldx = D; g1.W[0] = s.w1f[0]; g1.Wlo[0] = s.w1f[1]; g1.ldw = D; g1.bias[0] = b1; g1.M = B * N; g1.Nout = C1; g1.K = D;
    g1.Yf = s.P; g1.ldyf = C1; g1.xyz = xyz; g1.W1x[0] = W1; g1.ldw1x = 3 + D;
    PZ_TRY(launch_split_rowgemm(g1, st));
    TcGemm g2;
    g2.Xf = s.P; g2.ldx = C1; g2.Qf = s.Q; g2.rows = rows; g2.W[0] = s.w2[0]; g2.Wlo[0] = s.w2[1]; g2.ldw = C1; g2.bias[0] = b2; g2.M = (int)total;
    g2.Nout = C2; g2.K = C1; g2.epi = 1; g2.relu = 1; g2.Yf = out; g2.ldyf = C2;
    return launch_split_gather(g2, st);
  }
  if (precision == PZ_PREC_BF16) {
    // tensor-core path: P = feat W1[:,3:]^T + b1 + W1[:,0:3] xyz (row GEMM), then the gathered GEMM forms Q = W1[:,0:3] c
    // per stage in shared memory
    PZ_TRY(launch_cvt_bf16(feat, D, B * N, D, b.feat, D, st));
    PZ_TRY(launch_cvt_bf16(W1 + 3, 3 + D, C1, D, b.w1f, D, st));
    PZ_TRY(launch_cvt_bf16(W2, C1, C2, C1, b.w2, C1, st));
    TcGemm g1;
    g1.X = b.feat; g1.ldx = D; g1.W[0] = b.w1f; g1.ldw = D; g1.bias[0] = b1; g1.M = B * N; g1.Nout = C1; g1.K = D;
    g1.Yb = b.P; g1.ldyb = C1; g1.xyz = xyz; g1.W1x[0] = W1; g1.ldw1x = 3 + D;
    PZ_TRY(launch_tc_rowgemm(g1, st));
    TcGemm g2;
    g2.X = b.P; g2.ldx = C1; g2.rows = rows; g2.centers = new_xyz; g2.W1x[0] = W1; g2.ldw1x = 3 + D; g2.W[0] = b.w2; g2.ldw = C1; g2.bias[0] = b2; g2.M = (int)total;
    g2.Nout = C2; g2.K = C1; g2.epi = 1; g2.relu = 1; g2.Yf = out; g2.ldyf = C2;
    return launch_tc_gemm(g2, st);
  }
  GemmF32 g1;
  g1.A = feat; g1.lda = D; g1.W[0] = W1 + 3; g1.ldw = 3 + D; g1.Y = f.F; g1.ldy = C1; g1.M = B * N; g1.N = C1; g1.K = D;
  PZ_TRY(launch_gemm_f32(g1, st));
  GemmF32 g2;
  g2.A = f.F; g2.lda = C1; g2.rows = rows; g2.xyz = xyz; g2.centers = new_xyz; g2.W1[0] = W1; g2.b1[0] = b1;
  g2.ldw1 = 3 + D; g2.W[0] = W2; g2.bias[0] = b2; g2.ldw = C1; g2.Y = out; g2.ldy = C2; g2.M = (int)total;
  g2.N = C2; g2.K = C1; g2.relu = 1; g2.group = 32;
  return launch_gemm_f32(g2, st);
}
