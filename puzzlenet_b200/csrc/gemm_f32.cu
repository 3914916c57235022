// fp32 CUDA-core GEMM family for the "fp32-faithful" path (PZ_PREC_FP32):
//   Y[M,N] = epilogue(alpha * A[M,K] * W[N,K]^T + bias[N])
// Every nn.Linear of the encoder / heads (model5_b.py:447-475, :723-754) is this shape
// (activations [rows, in], weight [out, in]).  Tile 128 x BN x 16, 256 threads, 8 x (BN/16)
// register micro-tile split in two 4-wide halves so that shared-memory reads are
// conflict-free 128-bit loads; register-staged double buffering, one barrier per k-tile.
//
// A-operand sources:
//   PLAIN   rows of A
//   GATHER  layer 2 of the grouped shared MLP without materialising [B,S,K,3+D]
//           (pointnet_util.py:123-130 + model5_b.py:452-454):
//             A[r,k] = relu(F[rows[r],k] + b1[k] + W1[k,0:3] . (xyz[rows[r]] - centre[r/32]))
//           where F = feat * W1[:,3:]^T is layer 1 applied once per *source point* instead of
//           once per (group, neighbour) -- 16x fewer layer-1 MACs, same value up to fp32
//           summation order.
// Epilogues: bias(+relu), residual (Y = R + relu(..), model5_b.py:100), per-row-block bias
// table (boundary heads' global-feature half, model5_b.py:748-752) and max over groups of
// 32 / 128 consecutive rows (neighbourhood / point max-pool, model5_b.py:454, :475).
#include "pz_common.cuh"

namespace pz {

constexpr int BM = 128;
constexpr int BK = 16;
constexpr int GT = 256;  // threads

enum { A_PLAIN = 0, A_GATHER = 1 };
enum { EPI_STORE = 0, EPI_GROUPMAX = 1 };

template <int BN, int AMODE, int EPI, bool VEC_A, bool VEC_W>
__global__ void __launch_bounds__(GT, 2) gemm_f32_kernel(GemmF32 g) {
  constexpr int TN = BN / 16;  // 8 or 4 columns per thread
  constexpr int WPT = BN * BK / GT;  // W floats per thread per k-tile (8 or 4)
  __shared__ __align__(16) float tiles[2 * BK * BM + 2 * BK * BN];
  float (*As)[BK][BM] = reinterpret_cast<float (*)[BK][BM]>(tiles);
  float (*Bs)[BK][BN] = reinterpret_cast<float (*)[BK][BN]>(tiles + 2 * BK * BM);
  // GATHER: per-k (W1x0, W1x1, W1x2, b1) for the whole K, K <= 256
  __shared__ float4 w1s[AMODE == A_GATHER ? 256 : 1];
  float* red = tiles;  // group-max scratch [16][2][BN] aliases the A tiles after the main loop
  static_assert(16 * 2 * BN <= 2 * BK * BM, "reduction scratch must fit in the A tiles");

  const int t = threadIdx.x;
  const int tx = t & 15, ty = t >> 4;
  // (row tile, column tile) on the 1-D grid, column tile fastest: neighbouring CTAs share the rows of A in L2
  const int ntn = (g.N + BN - 1) / BN;
  const int mt = blockIdx.x / ntn;
  const int m0 = mt * BM, n0 = (blockIdx.x - mt * ntn) * BN;
  const int wset = g.rows_per_wset > 0 ? m0 / g.rows_per_wset : 0;
  // split-K: CTA z handles k in [z*ksplit, (z+1)*ksplit) and stores raw partial sums to Y + z*M*ldy
  const int kbeg = g.ksplit > 0 ? blockIdx.z * g.ksplit : 0;
  if (g.ksplit > 0) {
    g.K = min(g.K - kbeg, g.ksplit);
    g.Y += (size_t)blockIdx.z * g.M * g.ldy;
  }
  const float* __restrict__ W = g.W[wset];
  const float* __restrict__ bias = g.bias[wset];

  // ---- A loader state: thread -> (row, 8 consecutive k)
  const int a_row = t & 127, a_k = (t >> 7) * 8;
  const int am = m0 + a_row;
  const bool a_ok = am < g.M;
  const float* a_ptr = nullptr;
  float rx = 0.f, ry = 0.f, rz = 0.f;
  if (AMODE == A_PLAIN) {
    a_ptr = g.A + (size_t)(a_ok ? am : 0) * g.lda + kbeg;
  } else {
    const int src = a_ok ? g.rows[am] : 0;
    a_ptr = g.A + (size_t)src * g.lda;
    const float* c = g.centers + (size_t)(am >> 5) * 3;
    if (a_ok) {
      rx = __fsub_rn(g.xyz[(size_t)src * 3 + 0], c[0]);
      ry = __fsub_rn(g.xyz[(size_t)src * 3 + 1], c[1]);
      rz = __fsub_rn(g.xyz[(size_t)src * 3 + 2], c[2]);
    }
    const float* W1 = g.W1[wset];
    const float* b1 = g.b1[wset];
    for (int k = t; k < g.K; k += GT)
      w1s[k] = make_float4(W1[(size_t)k * g.ldw1], W1[(size_t)k * g.ldw1 + 1], W1[(size_t)k * g.ldw1 + 2], b1[k]);
    __syncthreads();
  }
  // ---- W loader state
  const int w_row = (BN == 128) ? (t & 127) : (t & 63);
  const int w_k = (BN == 128) ? (t >> 7) * 8 : (t >> 6) * 4;
  const int wn = n0 + w_row;
  const bool w_ok = wn < g.N;
  const float* w_ptr = W + (size_t)(w_ok ? wn : 0) * g.ldw + kbeg;

  float areg[8], wreg[WPT];
  auto load_tile = [&](int k0) {
    // A
    if (VEC_A) {
      if (a_ok && k0 + a_k < g.K) {  // K % 8 == 0 guaranteed by the dispatcher
        float4 v0 = *reinterpret_cast<const float4*>(a_ptr + k0 + a_k);
        float4 v1 = *reinterpret_cast<const float4*>(a_ptr + k0 + a_k + 4);
        areg[0] = v0.x; areg[1] = v0.y; areg[2] = v0.z; areg[3] = v0.w;
        areg[4] = v1.x; areg[5] = v1.y; areg[6] = v1.z; areg[7] = v1.w;
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) areg[i] = 0.f;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        int k = k0 + a_k + i;
        areg[i] = (a_ok && k < g.K) ? a_ptr[k] : 0.f;
      }
    }
    if (AMODE == A_GATHER) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        int k = k0 + a_k + i;
        if (a_ok && k < g.K) {
          float4 w = w1s[k];
          float v = areg[i] + w.w;
          v = fmaf(w.x, rx, v);
          v = fmaf(w.y, ry, v);
          v = fmaf(w.z, rz, v);
          areg[i] = fmaxf(v, 0.f);
        }
      }
    }
    // W
    if (VEC_W) {
      if (w_ok && k0 + w_k < g.K) {
        float4 v0 = *reinterpret_cast<const float4*>(w_ptr + k0 + w_k);
        wreg[0] = v0.x; wreg[1] = v0.y; wreg[2] = v0.z; wreg[3] = v0.w;
        if (WPT == 8) {
          float4 v1 = *reinterpret_cast<const float4*>(w_ptr + k0 + w_k + 4);
          wreg[WPT - 4] = v1.x; wreg[WPT - 3] = v1.y; wreg[WPT - 2] = v1.z; wreg[WPT - 1] = v1.w;
        }
      } else {
#pragma unroll
        for (int i = 0; i < WPT; ++i) wreg[i] = 0.f;
      }
    } else {
#pragma unroll
      for (int i = 0; i < WPT; ++i) {
        int k = k0 + w_k + i;
        wreg[i] = (w_ok && k < g.K) ? w_ptr[k] : 0.f;
      }
    }
  };
  auto store_tile = [&](int buf) {
#pragma unroll
    for (int i = 0; i < 8; ++i) As[buf][a_k + i][a_row] = areg[i];
#pragma unroll
    for (int i = 0; i < WPT; ++i) Bs[buf][w_k + i][w_row] = wreg[i];
  };

  float acc[8][TN];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  const int nk = (g.K + BK - 1) / BK;
  load_tile(0);
  store_tile(0);
  __syncthreads();
  for (int kt = 0; kt < nk; ++kt) {
    const int buf = kt & 1;
    if (kt + 1 < nk) load_tile((kt + 1) * BK);
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float a[8], b[TN];
      float4 a0 = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
      float4 a1 = *reinterpret_cast<const float4*>(&As[buf][k][64 + ty * 4]);
      a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w;
      a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
      float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
      b[0] = b0.x; b[1] = b0.y; b[2] = b0.z; b[3] = b0.w;
      if (TN == 8) {
        float4 b1v = *reinterpret_cast<const float4*>(&Bs[buf][k][(BN / 2) + tx * 4]);
        b[TN - 4] = b1v.x; b[TN - 3] = b1v.y; b[TN - 2] = b1v.z; b[TN - 1] = b1v.w;
      }
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (kt + 1 < nk) {
      store_tile(buf ^ 1);
      __syncthreads();
    }
  }

  // ---------------------------------------------------------------- epilogue
  // thread owns rows m0 + {ty*4+i, 64+ty*4+i} and cols n0 + {tx*4+j, BN/2+tx*4+j}
  auto col_of = [&](int j) { return n0 + ((TN == 8 && j >= 4) ? (BN / 2) + tx * 4 + (j - 4) : tx * 4 + j); };
  if (EPI == EPI_STORE) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int row = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
      if (row >= g.M) continue;
      const float* rb = g.rowbias ? g.rowbias + (size_t)(row / g.rb_rows) * g.N : nullptr;
#pragma unroll
      for (int jh = 0; jh < TN / 4; ++jh) {
        const int c0 = col_of(jh * 4);
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int col = c0 + j;
          float x = acc[i][jh * 4 + j] * g.alpha;
          if (col < g.N) {
            if (bias) x += bias[col];
            if (rb) x += rb[col];
            if (g.relu) x = fmaxf(x, 0.f);
            if (g.R) x += g.R[(size_t)row * g.ldr + col];
          }
          v[j] = x;
        }
        float* yp = g.Y + (size_t)row * g.ldy + c0;
        if (c0 + 3 < g.N && ((g.ldy & 3) == 0) && ((reinterpret_cast<uintptr_t>(g.Y) & 15) == 0)) {
          *reinterpret_cast<float4*>(yp) = make_float4(v[0], v[1], v[2], v[3]);
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (c0 + j < g.N) yp[j] = v[j];
        }
      }
    }
  } else {
    // max over groups of `group` consecutive rows (32 or 128); requires full M tiles.
    // red[ty][half][col]: max over the thread's 4 rows of each half.
    __syncthreads();  // every warp is done reading the operand tiles that `red` aliases
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      const int cl = (TN == 8 && j >= 4) ? (BN / 2) + tx * 4 + (j - 4) : tx * 4 + j;
      float mlo = fmaxf(fmaxf(acc[0][j], acc[1][j]), fmaxf(acc[2][j], acc[3][j]));
      float mhi = fmaxf(fmaxf(acc[4][j], acc[5][j]), fmaxf(acc[6][j], acc[7][j]));
      red[(ty * 2 + 0) * BN + cl] = mlo;
      red[(ty * 2 + 1) * BN + cl] = mhi;
    }
    __syncthreads();
    // rows of half h, thread-row ty are  h*64 + ty*4 .. +3  -> 32-row group index = h*2 + ty/8
    const int ngroups = BM / g.group;  // 4 or 1
    for (int o = t; o < ngroups * BN; o += GT) {
      const int gi = o / BN, cl = o - gi * BN;
      float m = -INFINITY;
      if (g.group == 32) {
        const int h = gi >> 1, tyb = (gi & 1) * 8;
#pragma unroll
        for (int u = 0; u < 8; ++u) m = fmaxf(m, red[((tyb + u) * 2 + h) * BN + cl]);
      } else {
        for (int u = 0; u < 32; ++u) m = fmaxf(m, red[u * BN + cl]);
      }
      const int col = n0 + cl;
      if (col < g.N) {
        float x = m * g.alpha;
        if (bias) x += bias[col];
        if (g.relu) x = fmaxf(x, 0.f);
        g.Y[(size_t)(m0 / g.group + gi) * g.ldy + col] = x;
      }
    }
  }
}

template <int BN, int AMODE, int EPI>
static int gemm_dispatch_vec(const GemmF32& g, cudaStream_t st) {
  const bool vec_a = (g.K % 8 == 0) && (g.lda % 4 == 0) && ((reinterpret_cast<uintptr_t>(g.A) & 15) == 0);
  bool vec_w = (g.K % 8 == 0) && (g.ldw % 4 == 0) && ((reinterpret_cast<uintptr_t>(g.W[0]) & 15) == 0);
  if (g.W[1]) vec_w = vec_w && ((reinterpret_cast<uintptr_t>(g.W[1]) & 15) == 0);
  const long long tiles = ((long long)g.M + BM - 1) / BM * ((g.N + BN - 1) / BN);   // <= 2^31 - 1: launch_gemm_f32
  dim3 grid((unsigned)tiles, 1, g.ksplit > 0 ? (g.K + g.ksplit - 1) / g.ksplit : 1);
  if (vec_a && vec_w)
    gemm_f32_kernel<BN, AMODE, EPI, true, true><<<grid, GT, 0, st>>>(g);
  else if (vec_a)
    gemm_f32_kernel<BN, AMODE, EPI, true, false><<<grid, GT, 0, st>>>(g);
  else if (vec_w)
    gemm_f32_kernel<BN, AMODE, EPI, false, true><<<grid, GT, 0, st>>>(g);
  else
    gemm_f32_kernel<BN, AMODE, EPI, false, false><<<grid, GT, 0, st>>>(g);
  PZ_LAUNCH_CHECK();
  return 0;
}

int launch_gemm_f32(const GemmF32& g, cudaStream_t st) {
  PZ_REQUIRE(g.A && g.W[0] && g.Y, PZ_ERR_ARG, "gemm_f32: null operand");
  PZ_REQUIRE(g.M > 0 && g.N > 0 && g.K > 0, PZ_ERR_ARG, "gemm_f32: bad shape %dx%dx%d", g.M, g.N, g.K);
  const int bn = g.N > 64 ? 128 : 64;
  PZ_REQUIRE(((long long)g.M + BM - 1) / BM * ((g.N + bn - 1) / bn) <= 0x7fffffff, PZ_ERR_UNSUPPORTED,
             "gemm_f32: M=%d N=%d needs more than 2^31 - 1 tiles", g.M, g.N);
  if (g.rows_per_wset > 0)
    PZ_REQUIRE(g.rows_per_wset % BM == 0 && g.W[(g.M - 1) / g.rows_per_wset] != nullptr, PZ_ERR_ARG,
               "gemm_f32: weight sets must cover whole %d-row tiles", BM);
  if (g.ksplit > 0)
    PZ_REQUIRE(g.ksplit % 8 == 0 && !g.rows && !g.group && !g.R && !g.rowbias && !g.bias[0] && !g.relu, PZ_ERR_ARG,
               "gemm_f32: split-K stores raw partial sums only");
  const bool gather = g.rows != nullptr;
  const bool gmax = g.group != 0;
  if (gmax)
    PZ_REQUIRE((g.group == 32 || g.group == 128) && g.M % BM == 0 && !g.R && !g.rowbias, PZ_ERR_ARG,
               "gemm_f32: group-max epilogue needs group in {32,128} and M %% 128 == 0");
  if (gather)
    PZ_REQUIRE(g.K <= 256 && g.xyz && g.centers && g.W1[0] && g.b1[0] && g.M % 32 == 0, PZ_ERR_ARG,
               "gemm_f32: gathered A needs K <= 256 and xyz/centers/W1/b1");
  const bool wide = bn == 128;
  if (gather) {
    if (gmax) return wide ? gemm_dispatch_vec<128, A_GATHER, EPI_GROUPMAX>(g, st) : gemm_dispatch_vec<64, A_GATHER, EPI_GROUPMAX>(g, st);
    return wide ? gemm_dispatch_vec<128, A_GATHER, EPI_STORE>(g, st) : gemm_dispatch_vec<64, A_GATHER, EPI_STORE>(g, st);
  }
  if (gmax) return wide ? gemm_dispatch_vec<128, A_PLAIN, EPI_GROUPMAX>(g, st) : gemm_dispatch_vec<64, A_PLAIN, EPI_GROUPMAX>(g, st);
  return wide ? gemm_dispatch_vec<128, A_PLAIN, EPI_STORE>(g, st) : gemm_dispatch_vec<64, A_PLAIN, EPI_STORE>(g, st);
}

}  // namespace pz
