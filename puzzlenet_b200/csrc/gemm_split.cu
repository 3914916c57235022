// tcgen05 GEMMs of the SPLIT path (PZ_PREC_SPLIT): the tensor-core path that meets the fp32 tolerances.
//
// Every operand x is carried as two fp16 planes, hi = fp16(x) and lo = fp16(x - hi) (22 mantissa bits together), and
// every product is three MMAs accumulated in fp32 in TMEM:
//     X W^T  ~=  Xhi Whi^T + Xhi Wlo^T + Xlo Whi^T            (the dropped Xlo Wlo^T term is ~2^-22 relative)
// which reproduces the reference's fp32 nn.Linear (model5_b.py:447-475) to ~1e-6 at three times the bf16 MMA count
// -- against ~40 times slower on the FFMA pipe (PZ_PREC_FP32).  fp16 rather than bf16 halves: 11 + 11 mantissa bits
// instead of 8 + 8 (measured against the oracle: rotation 2.5e-4 degree instead of 1.6e-3, north_star bound 0.01).
// Operands are scaled nowhere: |x| < 65504 is required of every activation (true of this network by four orders of
// magnitude); the fp16 conversions saturate instead of producing infinities.
//
// The kernels, all persistent and warp-specialised (epilogue warps / one MMA-issuing thread / producers) with an smem
// stage ring and a double-buffered TMEM accumulator:
//   split_rowgemm_pair_kernel : Y[row, ch] row-major GEMM on a CTA PAIR (tcgen05.mma.cta_group::2, M = 256 rows), operands
//                               by TMA, the CTA's weight half resident where it fits; every plain nn.Linear (layer 1 of the
//                               grouped MLPs over source points, q|k and v projections, out-projection with residual, tail)
//   split_rowgemm_kernel      : the one-CTA cp.async version (shapes that do not tile by 256 rows)
//   split_gather_kernel       : grouped-MLP layer 2 with the gathered operand relu(P[j] - Q[s]) formed IN REGISTERS from
//                               fp32 P rows (global -> registers -> swizzled st.shared per plane) and the max over the 32
//                               neighbours in the epilogue (pointnet_util.py:123-130 + model5_b.py:452-454, :459-461)
//   split_gather_pair_kernel  : the same for 256 output channels on a CTA pair: each gathered row is formed once for both
//                               128-channel blocks
#include <cuda.h>   // CUtensorMap (types only: the encoder is fetched with cudaGetDriverEntryPoint)
#include <cuda_fp16.h>
#include <stdlib.h>
#include <string.h>

#include "pz_common.cuh"
#include "tc_common.cuh"

namespace pz {

using namespace tc;

namespace {

constexpr int SG_THREADS = 13 * 32;
constexpr uint32_t TILE16K = 128 * 128;   // one [128 rows x 64 k] fp16 SWIZZLE_128B tile

// D=f32, A=B=f16 (format 0), both K-major, M=128, N=n
__host__ __device__ constexpr uint32_t make_idesc_f16(int n, int m = 128) {
  return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// two floats -> packed fp16 hi pair and packed fp16 lo pair (lo = fp16(x - hi)); saturating, so no infinities
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  uint32_t h;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h) : "f"(b), "f"(a));
  const __half2 hh = *reinterpret_cast<const __half2*>(&h);
  const float2 hf = __half22float2(hh);
  uint32_t l;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(l) : "f"(b - hf.y), "f"(a - hf.x));
  hi = h;
  lo = l;
}
__device__ __forceinline__ float2 join2(uint32_t hi, uint32_t lo) {
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&hi));
  const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&lo));
  return make_float2(a.x + b.x, a.y + b.y);
}

// the three MMAs of one K=16 step: hi*hi (+ accumulate flag), hi*lo, lo*hi
__device__ __forceinline__ void umma_split(uint32_t d, uint64_t a_hi, uint64_t a_lo, uint64_t b_hi, uint64_t b_lo,
                                           uint32_t idesc, uint32_t accumulate) {
  umma_bf16(d, a_hi, b_hi, idesc, accumulate);   // kind::f16 covers fp16 and bf16; the descriptor selects fp16
  umma_bf16(d, a_hi, b_lo, idesc, 1);
  umma_bf16(d, a_lo, b_hi, idesc, 1);
}

}  // namespace

// ============================================================================================== row-major GEMM
// Stage = [X hi 16 KB][X lo 16 KB][W hi NCOLS*128 B][W lo NCOLS*128 B]; thread = output row in the epilogue.
template <int NCOLS, int NST>
__global__ void __launch_bounds__(SG_THREADS, 1) split_rowgemm_kernel(const TcGemm g) {
  extern __shared__ __align__(1024) uint8_t srg_smem_raw[];
  const uint32_t smem_base = (smem_u32(srg_smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = srg_smem_raw + (smem_base - smem_u32(srg_smem_raw));
  constexpr int EPI = 8, PROD_THREADS = 128, ROWS = 128;
  constexpr uint32_t STAGE_X = 2 * TILE16K, W_PLANE = NCOLS * 128, STAGE = STAGE_X + 2 * W_PLANE;
  const uint32_t bars = smem_base + NST * STAGE;
  const uint32_t full_bar = bars, empty_bar = bars + 8 * NST, accf_bar = bars + 16 * NST, acce_bar = accf_bar + 16;
  const uint32_t tmem_slot = acce_bar + 16;
  const uint32_t chan_s = tmem_slot + 16;           // [NCOLS] float4 (w1x, w1y, w1z, bias)
  float4* chan = reinterpret_cast<float4*>(smem_gen + (chan_s - smem_base));
  int* colmax = reinterpret_cast<int*>(chan + NCOLS);   // [4 row quarters][NCOLS] order-preserving int images (Ymax epilogue)

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int kblocks = g.K / KB;
  const int nsets = (g.rows_per_wset > 0 && g.M > g.rows_per_wset) ? 2 : 1;
  const int row_tiles = g.M / ROWS, col_tiles = g.Nout / NCOLS;
  const int tiles_per_set = (row_tiles / nsets) * col_tiles;
  const int ctas_per_set = gridDim.x / nsets;
  const int wset = min((int)blockIdx.x / ctas_per_set, nsets - 1);
  const int rank_in_set = blockIdx.x - wset * ctas_per_set;
  const int step = (wset == nsets - 1) ? (int)gridDim.x - wset * ctas_per_set : ctas_per_set;
  const int tile_begin = wset * tiles_per_set;
  const __half* __restrict__ Whi = reinterpret_cast<const __half*>(g.W[wset]);
  const __half* __restrict__ Wlo = reinterpret_cast<const __half*>(g.Wlo[wset]);
  const __half* __restrict__ Xhi = reinterpret_cast<const __half*>(g.X);
  const __half* __restrict__ Xlo = reinterpret_cast<const __half*>(g.Xlo);
  const float* __restrict__ bias = g.bias[wset];

  if (tid == 0) {
    for (int s = 0; s < NST; ++s) {
      mbar_init(full_bar + 8 * s, PROD_THREADS);
      mbar_init(empty_bar + 8 * s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(accf_bar + 8 * b, 1);
      mbar_init(acce_bar + 8 * b, EPI * 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == EPI) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  pdl_enter();   // the prologue above touched no global memory
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  if (warp > EPI) {
    // ================================================= producers: cp.async the four planes of a stage
    const int pt = tid - (EPI + 1) * 32;
    uint32_t issued = 0, arrived = 0;
    for (int t = tile_begin + rank_in_set; t < tile_begin + tiles_per_set; t += step) {
      const int ct = t % col_tiles, rt = t / col_tiles;
      const int row0 = rt * ROWS, col0 = ct * NCOLS;
      for (int kb = 0; kb < kblocks; ++kb) {
        const uint32_t s = issued % NST, ph = (issued / NST) & 1;
        mbar_wait(empty_bar + 8 * s, ph ^ 1);
        const uint32_t st_addr = smem_base + s * STAGE;
        for (int id = pt; id < ROWS * 8; id += PROD_THREADS) {
          const int c = id & 7, r = id >> 3;
          const size_t off = (size_t)(row0 + r) * g.ldx + kb * KB + c * 8;
          cp_async16(st_addr + sw128(r, c), Xhi + off);
          cp_async16(st_addr + TILE16K + sw128(r, c), Xlo + off);
        }
        for (int id = pt; id < NCOLS * 8; id += PROD_THREADS) {
          const int c = id & 7, r = id >> 3;
          const size_t off = (size_t)(col0 + r) * g.ldw + kb * KB + c * 8;
          cp_async16(st_addr + STAGE_X + sw128(r, c), Whi + off);
          cp_async16(st_addr + STAGE_X + W_PLANE + sw128(r, c), Wlo + off);
        }
        cp_async_commit();
        ++issued;
        if (issued - arrived > (NST > 2 ? 2u : 1u)) {
          if (NST > 2) cp_async_wait<2>(); else cp_async_wait<1>();
          fence_proxy_async();
          mbar_arrive(full_bar + 8 * (arrived % NST));
          ++arrived;
        }
      }
    }
    cp_async_wait<0>();
    fence_proxy_async();
    while (arrived < issued) {
      mbar_arrive(full_bar + 8 * (arrived % NST));
      ++arrived;
    }
  } else if (warp == EPI) {
    // ================================================= MMA issuer
    if (lane == 0) {
      const uint32_t idesc = make_idesc_f16(NCOLS);
      uint32_t it = 0, tcn = 0;
      for (int t = tile_begin + rank_in_set; t < tile_begin + tiles_per_set; t += step, ++tcn) {
        const uint32_t buf = tcn & 1, aph = (tcn >> 1) & 1;
        mbar_wait(acce_bar + 8 * buf, aph ^ 1);
        tc_fence_after();
        for (int kb = 0; kb < kblocks; ++kb, ++it) {
          const uint32_t s = it % NST, ph = (it / NST) & 1;
          mbar_wait(full_bar + 8 * s, ph);
          tc_fence_after();
          const uint32_t st_addr = smem_base + s * STAGE;
          const uint64_t a_hi = make_desc(st_addr), a_lo = make_desc(st_addr + TILE16K);
          const uint64_t b_hi = make_desc(st_addr + STAGE_X), b_lo = make_desc(st_addr + STAGE_X + W_PLANE);
#pragma unroll
          for (int k4 = 0; k4 < KB / 16; ++k4)
            umma_split(tmem_base + buf * NCOLS, a_hi + 2 * k4, a_lo + 2 * k4, b_hi + 2 * k4, b_lo + 2 * k4, idesc,
                       (kb | k4) != 0);
          umma_commit(empty_bar + 8 * s);
        }
        umma_commit(accf_bar + 8 * buf);
      }
    }
  } else {
    // ================================================= epilogue: thread = row, 32 channels per TMEM load
    const int quarter = warp & 3, half = warp >> 2;
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    const bool has_xyz = g.xyz != nullptr, relu = g.relu != 0;
    const int nvalid = g.n_valid > 0 ? g.n_valid : g.Nout;
    __half* Ybhi = reinterpret_cast<__half*>(g.Yb);
    __half* Yblo = reinterpret_cast<__half*>(g.Yblo);
    __half* YThi = reinterpret_cast<__half*>(g.YT);
    __half* YTlo = reinterpret_cast<__half*>(g.YTlo);
    const __half* Rhi = reinterpret_cast<const __half*>(g.Rb);
    const __half* Rlo = reinterpret_cast<const __half*>(g.Rblo);
    uint32_t tcn = 0;
    int staged_ct = -1;
    for (int t = tile_begin + rank_in_set; t < tile_begin + tiles_per_set; t += step, ++tcn) {
      const int ct = t % col_tiles, rt = t / col_tiles;
      const int col0 = ct * NCOLS;
      const size_t row = (size_t)rt * ROWS + quarter * 32 + lane;
      if (ct != staged_ct) {
        asm volatile("bar.sync 1, 256;" ::: "memory");
        for (int c = tid; c < NCOLS; c += EPI * 32) {
          const int ch = col0 + c;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (ch < nvalid) {
            if (bias) v.w = bias[ch];
            if (has_xyz) {
              const float* wp = g.W1x[wset] + (size_t)ch * g.ldw1x;
              v.x = wp[0]; v.y = wp[1]; v.z = wp[2];
            }
          }
          chan[c] = v;
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
        staged_ct = ct;
      }
      float px = 0.f, py = 0.f, pz = 0.f;
      if (has_xyz) {
        const float* p = g.xyz + row * 3;
        px = p[0]; py = p[1]; pz = p[2];
      }
      const float* rbp = g.rowbias ? g.rowbias + (row / g.rb_rows) * g.rb_ld : nullptr;
      const uint32_t buf = tcn & 1, aph = (tcn >> 1) & 1;
      mbar_wait(accf_bar + 8 * buf, aph);
      tc_fence_after();
#pragma unroll 1
      for (int c32 = half; c32 < NCOLS / 32; c32 += 2) {
        const int cb = col0 + c32 * 32;
        if (cb >= nvalid) break;
        uint4 rh[4], rl[4];
        if (Rhi) {
          const uint4* ph = reinterpret_cast<const uint4*>(Rhi + row * g.ldrb + cb);
          const uint4* pl = reinterpret_cast<const uint4*>(Rlo + row * g.ldrb + cb);
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) { rh[q4] = ph[q4]; rl[q4] = pl[q4]; }
        }
        float v[32];
        tmem_ld32(tmem_base + lane_base + buf * NCOLS + c32 * 32, v);
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const float4 cc = chan[c32 * 32 + i];
          float x = v[i] + cc.w;
          if (has_xyz) x = fmaf(cc.x, px, fmaf(cc.y, py, fmaf(cc.z, pz, x)));
          v[i] = x;
        }
        if (rbp) {
#pragma unroll
          for (int q4 = 0; q4 < 8; ++q4) {
            const float4 b4 = *reinterpret_cast<const float4*>(rbp + cb + q4 * 4);
            v[q4 * 4] += b4.x; v[q4 * 4 + 1] += b4.y; v[q4 * 4 + 2] += b4.z; v[q4 * 4 + 3] += b4.w;
          }
        }
        if (relu) {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.f);
        }
        if (Rhi) {
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) {
            const uint32_t* hp = reinterpret_cast<const uint32_t*>(&rh[q4]);
            const uint32_t* lp = reinterpret_cast<const uint32_t*>(&rl[q4]);
#pragma unroll
            for (int h = 0; h < 4; ++h) {
              const float2 f = join2(hp[h], lp[h]);
              v[q4 * 8 + 2 * h] += f.x;
              v[q4 * 8 + 2 * h + 1] += f.y;
            }
          }
        }
        if (g.Rf) {
          const float4* rp = reinterpret_cast<const float4*>(g.Rf + row * g.ldrf + cb);
#pragma unroll
          for (int q4 = 0; q4 < 8; ++q4) {
            const float4 b4 = rp[q4];
            v[q4 * 4] += b4.x; v[q4 * 4 + 1] += b4.y; v[q4 * 4 + 2] += b4.z; v[q4 * 4 + 3] += b4.w;
          }
        }
        if (g.Ymax) {
          // column maxima over the tile's 128 rows: one redux.sync.max per channel over the warp's 32 rows on the
          // order-preserving integer image of the float, lane i keeps channel i; the four row quarters meet in smem
          int keep = 0;
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int o = __float_as_int(v[i]);
            const int m = __reduce_max_sync(0xffffffffu, o >= 0 ? o : o ^ 0x7fffffff);
            if (lane == i) keep = m;
          }
          colmax[quarter * NCOLS + c32 * 32 + lane] = keep;
        }
        if (YThi) {
          // transposed planes, per block of t_rows rows (one cloud): YT[(blk * Nout + ch) * t_rows + row_in_blk];
          // the 32 lanes of a warp are 32 consecutive rows -> 64 contiguous bytes per channel and plane
          const size_t blk = row / g.t_rows, rin = row - blk * g.t_rows;
          __half* dh = YThi + (blk * g.Nout + cb) * g.t_rows + rin;
          __half* dl = YTlo + (blk * g.Nout + cb) * g.t_rows + rin;
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            uint32_t hi, lo;
            split2(v[i], v[i + 1], hi, lo);
            const __half2 h2 = *reinterpret_cast<const __half2*>(&hi), l2 = *reinterpret_cast<const __half2*>(&lo);
            dh[(size_t)i * g.t_rows] = __low2half(h2);
            dh[(size_t)(i + 1) * g.t_rows] = __high2half(h2);
            dl[(size_t)i * g.t_rows] = __low2half(l2);
            dl[(size_t)(i + 1) * g.t_rows] = __high2half(l2);
          }
        }
        if (Ybhi) {
          uint4* yh = reinterpret_cast<uint4*>(Ybhi + row * g.ldyb + cb);
          uint4* yl = reinterpret_cast<uint4*>(Yblo + row * g.ldyb + cb);
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) {
            uint4 oh, ol;
            split2(v[q4 * 8 + 0], v[q4 * 8 + 1], oh.x, ol.x);
            split2(v[q4 * 8 + 2], v[q4 * 8 + 3], oh.y, ol.y);
            split2(v[q4 * 8 + 4], v[q4 * 8 + 5], oh.z, ol.z);
            split2(v[q4 * 8 + 6], v[q4 * 8 + 7], oh.w, ol.w);
            yh[q4] = oh;
            yl[q4] = ol;
          }
        }
        if (g.Yf) {
          float4* yp = reinterpret_cast<float4*>(g.Yf + row * g.ldyf + cb);
#pragma unroll
          for (int q4 = 0; q4 < 8; ++q4) yp[q4] = make_float4(v[q4 * 4], v[q4 * 4 + 1], v[q4 * 4 + 2], v[q4 * 4 + 3]);
        }
      }
      tc_fence_before();
      mbar_arrive(acce_bar + 8 * buf);
      if (g.Ymax) {   // Ymax[row tile, ch] = max over the tile's rows (the caller folds the tiles of a cloud)
        asm volatile("bar.sync 1, 256;" ::: "memory");
        for (int c = tid; c < NCOLS && col0 + c < nvalid; c += EPI * 32) {
          const int m = max(max(colmax[c], colmax[NCOLS + c]), max(colmax[2 * NCOLS + c], colmax[3 * NCOLS + c]));
          g.Ymax[(size_t)rt * g.ldmax + col0 + c] = __int_as_float(m >= 0 ? m : m ^ 0x7fffffff);
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");   // colmax is rewritten by the next tile
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == EPI) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

template <int NCOLS, int NST>
static int split_rowgemm_launch(const TcGemm& g, cudaStream_t st) {
  const size_t smem = 1024 + (size_t)NST * (2 * TILE16K + 2 * NCOLS * 128) + 8 * (2 * NST + 4) + 32 + (size_t)NCOLS * 32;
  static_assert(1024 + (size_t)NST * (2 * TILE16K + 2 * NCOLS * 128) + 8 * (2 * NST + 4) + 32 + (size_t)NCOLS * 32 <= 232448,
                "split_rowgemm: shared memory budget");
  auto kern = split_rowgemm_kernel<NCOLS, NST>;
  PZ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int nsets = (g.rows_per_wset > 0 && g.M > g.rows_per_wset) ? 2 : 1;
  const int tiles = (g.M / 128) * (g.Nout / NCOLS);
  int grid = tiles < kNumSMs ? tiles : kNumSMs;
  if (nsets == 2 && (grid & 1)) --grid;
  if (grid < nsets) grid = nsets;
  PZ_CUDA(launch_pdl(kern, dim3(grid), dim3(SG_THREADS), smem, st, g));
  PZ_LAUNCH_CHECK();
  return 0;
}

// ============================================================================================== row-major GEMM, CTA pair
// The same GEMM on a CTA pair (tcgen05.mma.cta_group::2, M = 256 rows): every CTA streams the X planes of ITS 128 rows
// and holds HALF of the output channels' weights -- the pair shares the B operand, so a CTA moves half the weight bytes
// per flop.  RESIDENT (Nout == NCOLS and both planes of the CTA's weight half fit beside the stages: the attention
// projections, P1, P2): the weights are loaded once per CTA and only X streams (32 KB per k-block instead of 96 KB, the
// compulsory read of X); otherwise (the encoder tail) a stage carries X + the CTA's weight half of the column tile
// (64 KB).  Barrier protocol as in split_gather_pair_kernel: CTA-local full barriers, two relay threads in the peer CTA
// (stage full / accumulator drained) forward them to the leader with cluster-scope arrives, multicast commits back.
constexpr int RP_THREADS = 11 * 32;   // 8 epilogue warps, MMA issuer (leader) / stage relay (peer), accumulator relay, TMA producer

// operand tiles arrive by TMA (cp.async.bulk.tensor): one instruction per [rows x 64 k] SWIZZLE_128B tile, completion
// counted in bytes on the stage's mbarrier.  With cp.async the 128 producer threads needed ~250 instructions each per
// 64 KB stage and a stage took 3.4 us from issue to arrival (the tail GEMM ran at one k-block per 1.65 us against 0.78 us
// of MMAs); an L2-resident stream reaches 15-19 TB/s on this chip (scripts/l2_probe.cu), so the copy engine is not the limit.
struct alignas(64) RpMaps {
  CUtensorMap x[2];      // X hi / lo planes: [M, K] fp16, boxes of [128 rows x 64 k]
  CUtensorMap w[2][2];   // [weight set][hi / lo]: [Nout, K] fp16, boxes of [HALF rows x 64 k]
};
__device__ __forceinline__ void rp_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void rp_tma_load(uint32_t dst, const CUtensorMap* tm, int c0, int c1, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1) : "memory");
}

// timeline stamps of the first CTA pair (diagnostics, pz_profile_attention_timeline): globaltimer in ns, slot base
// 2048 + 512 * cluster rank; layout: 0 entry, 1 after cluster sync, 2 weights landed, 16+2j / 17+2j producer issue /
// arrive of job j, 128+j MMAs of job j issued, 192+2t / 193+2t epilogue of tile t sees the accumulator / is done, 3 exit
__device__ __forceinline__ void rp_stamp(long long* prof, uint32_t crank, int slot) {
  if (prof != nullptr && blockIdx.x < 2) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    prof[2048 + 512 * (int)crank + slot] = (long long)t;
  }
}

template <int NCOLS, int NST, bool RESIDENT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(RP_THREADS, 1) split_rowgemm_pair_kernel(const TcGemm g, const __grid_constant__ RpMaps maps) {
  extern __shared__ __align__(1024) uint8_t srp_smem_raw[];
  const uint32_t smem_base = smem_u32(srp_smem_raw);
  if ((smem_base & 1023u) != 0) __trap();   // no alignment pad is budgeted (see split_gather_pair_kernel)
  uint8_t* smem_gen = srp_smem_raw;
  constexpr int EPI = 8, ROWS = 128, HALF = NCOLS / 2;
  constexpr uint32_t STAGE_X = 2 * TILE16K, W_TILE = HALF * 128, STAGE = STAGE_X + (RESIDENT ? 0u : 2 * W_TILE);
  const int kblocks = g.K / KB;
  const uint32_t resident = RESIDENT ? (uint32_t)kblocks * 2 * W_TILE : 0u;   // per k-block [hi tile][lo tile]
  const uint32_t stages_base = smem_base + resident;
  const uint32_t bars = stages_base + NST * STAGE;
  const uint32_t full_bar = bars, empty_bar = bars + 8 * NST, pfull_bar = bars + 16 * NST;
  const uint32_t accf_bar = bars + 24 * NST, acce_bar = accf_bar + 16, pacce_bar = acce_bar + 16;
  const uint32_t w_bar = pacce_bar + 16;                        // resident weights of THIS CTA have landed
  const uint32_t tmem_slot = w_bar + 8;
  const uint32_t chan_s = (tmem_slot + 16 + 15) & ~15u;
  const bool has_xyz = g.xyz != nullptr;
  // per channel: (w1x, w1y, w1z, bias) when the layer has an xyz term, else the bias alone
  float4* chan4 = reinterpret_cast<float4*>(smem_gen + (chan_s - smem_base));
  float* chan1 = reinterpret_cast<float*>(chan4);
  const uint32_t colmax_s = chan_s + (has_xyz ? NCOLS * 16 : NCOLS * 4);
  int* colmax = reinterpret_cast<int*>(smem_gen + (colmax_s - smem_base));
  const uint32_t stage_s = (colmax_s + (g.Ymax ? NCOLS * 16 : 0) + 127) & ~127u;   // 8 x 4 KB epilogue staging tiles (when something is stored / a residual read)

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t crank = cluster_ctarank();
  if (tid == 0) rp_stamp(g.prof, crank, 0);
  const int npairs = gridDim.x >> 1, pair = blockIdx.x >> 1;
  const int nsets = (g.rows_per_wset > 0 && g.M > g.rows_per_wset) ? 2 : 1;
  const int row_tiles = g.M / (2 * ROWS), col_tiles = g.Nout / NCOLS;
  const int tiles_per_set = (row_tiles / nsets) * col_tiles;
  const int pairs_per_set = npairs / nsets;
  const int wset = min(pair / pairs_per_set, nsets - 1);
  const int rank_in_set = pair - wset * pairs_per_set;
  const int step = (wset == nsets - 1) ? npairs - wset * pairs_per_set : pairs_per_set;
  const int tile_begin = wset * tiles_per_set;
  const float* __restrict__ bias = g.bias[wset];

  if (tid == 0) {
    for (int s = 0; s < NST; ++s) {
      mbar_init(full_bar + 8 * s, 1);          // the producer's expect_tx arrival + the stage's bytes
      mbar_init(empty_bar + 8 * s, 1);
      mbar_init(pfull_bar + 8 * s, 1);     // leader: the peer's stage s is full
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(accf_bar + 8 * b, 1);
      mbar_init(acce_bar + 8 * b, EPI * 32);
      mbar_init(pacce_bar + 8 * b, 1);     // leader: the peer has drained accumulator b
    }
    mbar_init(w_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == EPI) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  pdl_enter();   // the prologue above touched no global memory
  tc_fence_before();
  cluster_sync_all();        // barriers initialised and TMEM allocated in both CTAs
  tc_fence_after();
  if (tid == 0) rp_stamp(g.prof, crank, 1);
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  if (warp >= EPI + 2) {
    // ================================================= producer: ONE thread issues the TMA loads of this CTA's tiles
    if (lane == 0) {
      const CUtensorMap* tx_hi = &maps.x[0];
      const CUtensorMap* tx_lo = &maps.x[1];
      const CUtensorMap* tw_hi = &maps.w[wset][0];
      const CUtensorMap* tw_lo = &maps.w[wset][1];
      if (RESIDENT) {   // this CTA's half of the output channels, both planes, one [HALF ch x 64 k] tile per k-block and plane
        rp_expect_tx(w_bar, (uint32_t)kblocks * 2 * W_TILE);
        for (int kb = 0; kb < kblocks; ++kb) {
          rp_tma_load(smem_base + (uint32_t)kb * 2 * W_TILE, tw_hi, kb * KB, (int)crank * HALF, w_bar);
          rp_tma_load(smem_base + (uint32_t)kb * 2 * W_TILE + W_TILE, tw_lo, kb * KB, (int)crank * HALF, w_bar);
        }
      }
      uint32_t issued = 0;
      for (int t = tile_begin + rank_in_set; t < tile_begin + tiles_per_set; t += step) {
        const int ct = t % col_tiles, rt = t / col_tiles;
        const int row0 = rt * 2 * ROWS + (int)crank * ROWS, col0 = ct * NCOLS + (int)crank * HALF;
        for (int kb = 0; kb < kblocks; ++kb, ++issued) {
          const uint32_t s = issued % NST, ph = (issued / NST) & 1;
          mbar_wait(empty_bar + 8 * s, ph ^ 1);
          const uint32_t st_addr = stages_base + s * STAGE;
          if (issued < 48) rp_stamp(g.prof, crank, 16 + 2 * (int)issued);
          rp_expect_tx(full_bar + 8 * s, STAGE);
          rp_tma_load(st_addr, tx_hi, kb * KB, row0, full_bar + 8 * s);
          rp_tma_load(st_addr + TILE16K, tx_lo, kb * KB, row0, full_bar + 8 * s);
          if (!RESIDENT) {
            rp_tma_load(st_addr + STAGE_X, tw_hi, kb * KB, col0, full_bar + 8 * s);
            rp_tma_load(st_addr + STAGE_X + W_TILE, tw_lo, kb * KB, col0, full_bar + 8 * s);
          }
        }
      }
    }
  } else if (warp == EPI) {
    if (crank == 0 && lane == 0) {
      // ================================================= MMA issuer: one thread of the leader CTA
      const uint32_t idesc = make_idesc_f16(NCOLS, 256);
      uint32_t it = 0, tcn = 0;
      if (RESIDENT) mbar_wait(w_bar, 0);
      rp_stamp(g.prof, crank, 2);
      for (int t = tile_begin + rank_in_set; t < tile_begin + tiles_per_set; t += step, ++tcn) {
        const uint32_t buf = tcn & 1, aph = (tcn >> 1) & 1;
        mbar_wait(acce_bar + 8 * buf, aph ^ 1);
        mbar_wait_cluster(pacce_bar + 8 * buf, aph ^ 1);
        tc_fence_after();
        for (int kb = 0; kb < kblocks; ++kb, ++it) {
          const uint32_t s = it % NST, ph = (it / NST) & 1;
          mbar_wait(full_bar + 8 * s, ph);
          mbar_wait_cluster(pfull_bar + 8 * s, ph);
          tc_fence_after();
          const uint32_t st_addr = stages_base + s * STAGE;
          const uint32_t w_addr = RESIDENT ? smem_base + (uint32_t)kb * 2 * W_TILE : st_addr + STAGE_X;
          const uint64_t a_hi = make_desc(st_addr), a_lo = make_desc(st_addr + TILE16K);
          const uint64_t b_hi = make_desc(w_addr), b_lo = make_desc(w_addr + W_TILE);
#pragma unroll
          for (int k4 = 0; k4 < KB / 16; ++k4) {
            const uint32_t d = tmem_base + buf * NCOLS;
            umma_f16_pair(d, a_hi + 2 * k4, b_hi + 2 * k4, idesc, (kb | k4) != 0);
            umma_f16_pair(d, a_hi + 2 * k4, b_lo + 2 * k4, idesc, 1);
            umma_f16_pair(d, a_lo + 2 * k4, b_hi + 2 * k4, idesc, 1);
          }
          umma_commit_pair(empty_bar + 8 * s);
          if (it < 64) rp_stamp(g.prof, crank, 128 + (int)it);
        }
        umma_commit_pair(accf_bar + 8 * buf);
      }
    } else if (crank == 1 && lane == 0) {
      // ================================================= stage relay of the peer CTA
      const uint32_t pfull_remote = mapa_shared(pfull_bar, 0);
      uint32_t jobs = 0;
      for (int t = tile_begin + rank_in_set; t < tile_begin + tiles_per_set; t += step) jobs += (uint32_t)kblocks;
      if (RESIDENT) mbar_wait(w_bar, 0);   // the first forwarded stage also vouches for this CTA's weights
      for (uint32_t it = 0; it < jobs; ++it) {
        const uint32_t s = it % NST, ph = (it / NST) & 1;
        mbar_wait(full_bar + 8 * s, ph);
        mbar_arrive_cluster(pfull_remote + 8 * s);
      }
    }
  } else if (warp == EPI + 1) {
    if (crank == 1 && lane == 0) {
      // ================================================= accumulator relay of the peer CTA
      const uint32_t pacce_remote = mapa_shared(pacce_bar, 0);
      uint32_t tcn = 0;
      for (int t = tile_begin + rank_in_set; t < tile_begin + tiles_per_set; t += step, ++tcn) {
        const uint32_t buf = tcn & 1, aph = (tcn >> 1) & 1;
        mbar_wait(acce_bar + 8 * buf, aph);
        mbar_arrive_cluster(pacce_remote + 8 * buf);
      }
    }
  } else {
    // ================================================= epilogue: thread = row of this CTA's 128 (its TMEM lane), 32
    // channels per TMEM load.  Global traffic is COALESCED through a 4 KB per-warp staging tile: a thread owns a row, so
    // direct 16-byte accesses touch 32 cache lines per warp instruction (measured: 46 us per launch against a 16 us HBM
    // floor, L1 wavefronts 48 %); instead the warp's [32 rows x 32 ch] block goes through shared memory (XOR-swizzled
    // 16-byte pieces, conflict-free both ways) and leaves / arrives as whole 64- or 128-byte row segments.  The residual
    // block of the NEXT chunk is prefetched into registers while the current one is finished.
    const int quarter = warp & 3, half = warp >> 2;
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    const bool relu = g.relu != 0;
    const int nvalid = g.n_valid > 0 ? g.n_valid : g.Nout;
    __half* Ybhi = reinterpret_cast<__half*>(g.Yb);
    __half* Yblo = reinterpret_cast<__half*>(g.Yblo);
    __half* YThi = reinterpret_cast<__half*>(g.YT);
    __half* YTlo = reinterpret_cast<__half*>(g.YTlo);
    const __half* Rhi = reinterpret_cast<const __half*>(g.Rb);
    const __half* Rlo = reinterpret_cast<const __half*>(g.Rblo);
    const uint32_t stg = stage_s + (uint32_t)warp * 4096;     // this warp's staging tile
    // 16-bit tiles: two planes of [32 rows][64 B]; piece p (8 channels) of row r sits at r*64 + ((p ^ ((r>>1)&3)) << 4)
    const int cr = lane >> 2, cp = lane & 3;                    // coalesced role: row 8j + cr, piece cp
    const uint32_t own16 = stg + (uint32_t)lane * 64, sw_own16 = (uint32_t)((lane >> 1) & 3);
    // fp32 tiles: [32 rows][128 B]; piece p (4 channels) of row r at r*128 + ((p ^ (r&7)) << 4)
    const int fr = lane >> 3, fp = lane & 7;                    // coalesced role: row 4j + fr, piece fp
    uint32_t tcn = 0;
    int staged_ct = -1;
    for (int t = tile_begin + rank_in_set; t < tile_begin + tiles_per_set; t += step, ++tcn) {
      const int ct = t % col_tiles, rt = (t / col_tiles) * 2 + (int)crank;   // rt: this CTA's 128-row tile
      const int col0 = ct * NCOLS;
      const size_t rowbase = (size_t)rt * ROWS + quarter * 32;
      const size_t row = rowbase + lane;
      if (ct != staged_ct) {
        asm volatile("bar.sync 1, 256;" ::: "memory");
        for (int c = tid; c < NCOLS; c += EPI * 32) {
          const int ch = col0 + c;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (ch < nvalid) {
            if (bias) v.w = bias[ch];
            if (has_xyz) {
              const float* wp = g.W1x[wset] + (size_t)ch * g.ldw1x;
              v.x = wp[0]; v.y = wp[1]; v.z = wp[2];
            }
          }
          if (has_xyz) chan4[c] = v; else chan1[c] = v.w;
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
        staged_ct = ct;
      }
      float px = 0.f, py = 0.f, pz = 0.f;
      if (has_xyz) {
        const float* p = g.xyz + row * 3;
        px = p[0]; py = p[1]; pz = p[2];
      }
      const float* rbp = g.rowbias ? g.rowbias + (row / g.rb_rows) * g.rb_ld : nullptr;
      uint4 pre[8];
      auto r_prefetch = [&](int cb) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const size_t off = (rowbase + 8 * j + cr) * g.ldrb + cb + cp * 8;
          pre[j] = *reinterpret_cast<const uint4*>(Rhi + off);
          pre[4 + j] = *reinterpret_cast<const uint4*>(Rlo + off);
        }
      };
      if (Rhi && col0 + half * 32 < nvalid) r_prefetch(col0 + half * 32);
      const uint32_t buf = tcn & 1, aph = (tcn >> 1) & 1;
      mbar_wait(accf_bar + 8 * buf, aph);
      tc_fence_after();
      if (tid == 0 && tcn < 32) rp_stamp(g.prof, crank, 192 + 2 * (int)tcn);
#pragma unroll 1
      for (int c32 = half; c32 < NCOLS / 32; c32 += 2) {
        const int cb = col0 + c32 * 32;
        if (cb >= nvalid) break;
        if (Rhi) {   // the prefetched residual block -> staging (coalesced role)
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int r = 8 * j + cr;
            const uint32_t a = stg + (uint32_t)r * 64 + (uint32_t)((cp ^ ((r >> 1) & 3)) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(pre[j].x), "r"(pre[j].y), "r"(pre[j].z), "r"(pre[j].w) : "memory");
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a + 2048), "r"(pre[4 + j].x), "r"(pre[4 + j].y), "r"(pre[4 + j].z), "r"(pre[4 + j].w) : "memory");
          }
          __syncwarp();
        }
        float v[32];
        tmem_ld32(tmem_base + lane_base + buf * NCOLS + c32 * 32, v);
        if (has_xyz) {
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const float4 cc = chan4[c32 * 32 + i];
            v[i] = fmaf(cc.x, px, fmaf(cc.y, py, fmaf(cc.z, pz, v[i] + cc.w)));
          }
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] += chan1[c32 * 32 + i];
        }
        if (rbp) {
#pragma unroll
          for (int q4 = 0; q4 < 8; ++q4) {
            const float4 b4 = *reinterpret_cast<const float4*>(rbp + cb + q4 * 4);
            v[q4 * 4] += b4.x; v[q4 * 4 + 1] += b4.y; v[q4 * 4 + 2] += b4.z; v[q4 * 4 + 3] += b4.w;
          }
        }
        if (relu) {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.f);
        }
        if (Rhi) {   // own row of the staged residual block
#pragma unroll
          for (int p4 = 0; p4 < 4; ++p4) {
            uint4 h, l;
            const uint32_t a = own16 + (((uint32_t)p4 ^ sw_own16) << 4);
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(h.x), "=r"(h.y), "=r"(h.z), "=r"(h.w) : "r"(a));
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(l.x), "=r"(l.y), "=r"(l.z), "=r"(l.w) : "r"(a + 2048));
            const uint32_t* hp = reinterpret_cast<const uint32_t*>(&h);
            const uint32_t* lp = reinterpret_cast<const uint32_t*>(&l);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 f = join2(hp[e], lp[e]);
              v[p4 * 8 + 2 * e] += f.x;
              v[p4 * 8 + 2 * e + 1] += f.y;
            }
          }
          __syncwarp();
          if (c32 + 2 < NCOLS / 32 && cb + 64 < nvalid) r_prefetch(cb + 64);   // next chunk of this warp
        }
        if (g.Rf) {
          const float4* rp = reinterpret_cast<const float4*>(g.Rf + row * g.ldrf + cb);
#pragma unroll
          for (int q4 = 0; q4 < 8; ++q4) {
            const float4 b4 = rp[q4];
            v[q4 * 4] += b4.x; v[q4 * 4 + 1] += b4.y; v[q4 * 4 + 2] += b4.z; v[q4 * 4 + 3] += b4.w;
          }
        }
        if (g.Ymax) {
          int keep = 0;
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int o = __float_as_int(v[i]);
            const int m = __reduce_max_sync(0xffffffffu, o >= 0 ? o : o ^ 0x7fffffff);
            if (lane == i) keep = m;
          }
          colmax[quarter * NCOLS + c32 * 32 + lane] = keep;
        }
        if (YThi) {
          const size_t blk = row / g.t_rows, rin = row - blk * g.t_rows;
          __half* dh = YThi + (blk * g.Nout + cb) * g.t_rows + rin;
          __half* dl = YTlo + (blk * g.Nout + cb) * g.t_rows + rin;
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            uint32_t hi, lo;
            split2(v[i], v[i + 1], hi, lo);
            const __half2 h2 = *reinterpret_cast<const __half2*>(&hi), l2 = *reinterpret_cast<const __half2*>(&lo);
            dh[(size_t)i * g.t_rows] = __low2half(h2);
            dh[(size_t)(i + 1) * g.t_rows] = __high2half(h2);
            dl[(size_t)i * g.t_rows] = __low2half(l2);
            dl[(size_t)(i + 1) * g.t_rows] = __high2half(l2);
          }
        }
        if (Ybhi) {
#pragma unroll
          for (int p4 = 0; p4 < 4; ++p4) {
            uint4 oh, ol;
            split2(v[p4 * 8 + 0], v[p4 * 8 + 1], oh.x, ol.x);
            split2(v[p4 * 8 + 2], v[p4 * 8 + 3], oh.y, ol.y);
            split2(v[p4 * 8 + 4], v[p4 * 8 + 5], oh.z, ol.z);
            split2(v[p4 * 8 + 6], v[p4 * 8 + 7], oh.w, ol.w);
            const uint32_t a = own16 + (((uint32_t)p4 ^ sw_own16) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(oh.x), "r"(oh.y), "r"(oh.z), "r"(oh.w) : "memory");
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a + 2048), "r"(ol.x), "r"(ol.y), "r"(ol.z), "r"(ol.w) : "memory");
          }
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int r = 8 * j + cr;
            const uint32_t a = stg + (uint32_t)r * 64 + (uint32_t)((cp ^ ((r >> 1) & 3)) << 4);
            uint4 h, l;
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(h.x), "=r"(h.y), "=r"(h.z), "=r"(h.w) : "r"(a));
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(l.x), "=r"(l.y), "=r"(l.z), "=r"(l.w) : "r"(a + 2048));
            const size_t off = (rowbase + r) * g.ldyb + cb + cp * 8;
            *reinterpret_cast<uint4*>(Ybhi + off) = h;
            *reinterpret_cast<uint4*>(Yblo + off) = l;
          }
          __syncwarp();
        }
        if (g.Yf) {
#pragma unroll
          for (int p8 = 0; p8 < 8; ++p8) {
            const uint32_t a = stg + (uint32_t)lane * 128 + (uint32_t)((p8 ^ (lane & 7)) << 4);
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v[p8 * 4]), "f"(v[p8 * 4 + 1]), "f"(v[p8 * 4 + 2]), "f"(v[p8 * 4 + 3]) : "memory");
          }
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int r = 4 * j + fr;
            const uint32_t a = stg + (uint32_t)r * 128 + (uint32_t)((fp ^ (r & 7)) << 4);
            float4 o;
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(o.x), "=f"(o.y), "=f"(o.z), "=f"(o.w) : "r"(a));
            *reinterpret_cast<float4*>(g.Yf + (rowbase + r) * g.ldyf + cb + fp * 4) = o;
          }
          __syncwarp();
        }
      }
      tc_fence_before();
      mbar_arrive(acce_bar + 8 * buf);
      if (tid == 0 && tcn < 32) rp_stamp(g.prof, crank, 193 + 2 * (int)tcn);
      if (g.Ymax) {   // Ymax[row tile, ch] = max over the tile's rows (the caller folds the tiles of a cloud)
        asm volatile("bar.sync 1, 256;" ::: "memory");
        for (int c = tid; c < NCOLS && col0 + c < nvalid; c += EPI * 32) {
          const int m = max(max(colmax[c], colmax[NCOLS + c]), max(colmax[2 * NCOLS + c], colmax[3 * NCOLS + c]));
          g.Ymax[(size_t)rt * g.ldmax + col0 + c] = __int_as_float(m >= 0 ? m : m ^ 0x7fffffff);
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");   // colmax is rewritten by the next tile
      }
    }
  }
  tc_fence_before();
  cluster_sync_all();
  if (tid == 0) rp_stamp(g.prof, crank, 3);
  if (warp == EPI) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

static size_t split_rowgemm_pair_smem(const TcGemm& g, int ncols, int nst, bool resident) {
  const size_t stage = 2 * TILE16K + (resident ? 0 : (size_t)ncols * 128);
  const bool staging = g.Yb || g.Yf || g.Rb;
  return (resident ? (size_t)(g.K / KB) * ncols * 128 : 0) + (size_t)nst * stage + 8 * (3 * nst + 7) + 48 +
         (size_t)ncols * (g.xyz ? 16 : 4) + (g.Ymax ? (size_t)ncols * 16 : 0) + 128 + (staging ? 8 * 4096 : 0);
}

// 2-D fp16 view [rows, cols] with a row stride of ld elements, traversed in [box_rows x 64] SWIZZLE_128B boxes
static int rp_make_map(const void* ptr, int ld, size_t rows, int cols, int box_rows, CUtensorMap* out) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn encode = [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      fn = nullptr;
    return reinterpret_cast<EncodeFn>(fn);
  }();
  PZ_REQUIRE(encode != nullptr, PZ_ERR_UNSUPPORTED, "split_rowgemm: the driver does not export cuTensorMapEncodeTiled");
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(__half)};
  const cuuint32_t box[2] = {64, (cuuint32_t)box_rows}, estr[2] = {1, 1};
  const CUresult r = encode(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  PZ_REQUIRE(r == CUDA_SUCCESS, PZ_ERR_ARG, "split_rowgemm: cuTensorMapEncodeTiled failed (%d)", (int)r);
  return 0;
}

template <int NCOLS, int NST, bool RESIDENT>
static int split_rowgemm_pair_launch(const TcGemm& g, cudaStream_t st) {
  const size_t smem = split_rowgemm_pair_smem(g, NCOLS, NST, RESIDENT);
  PZ_REQUIRE(smem <= 232448, PZ_ERR_UNSUPPORTED, "split_rowgemm (pair): needs %zu B of shared memory", smem);
  auto kern = split_rowgemm_pair_kernel<NCOLS, NST, RESIDENT>;
  PZ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int nsets = (g.rows_per_wset > 0 && g.M > g.rows_per_wset) ? 2 : 1;
  const int tiles_per_set = (g.M / 256 / nsets) * (g.Nout / NCOLS);
  int per = (kNumSMs / 2) / nsets;
  if (per > tiles_per_set) per = tiles_per_set;
  if (per < 1) per = 1;
  RpMaps maps;
  PZ_TRY(rp_make_map(g.X, g.ldx, (size_t)g.M, g.K, 128, &maps.x[0]));
  PZ_TRY(rp_make_map(g.Xlo, g.ldx, (size_t)g.M, g.K, 128, &maps.x[1]));
  for (int ws = 0; ws < 2; ++ws) {
    const int src = ws < nsets ? ws : 0;   // an unused second set repeats the first: every map handed over is valid
    PZ_TRY(rp_make_map(g.W[src], g.ldw, (size_t)g.Nout, g.K, NCOLS / 2, &maps.w[ws][0]));
    PZ_TRY(rp_make_map(g.Wlo[src], g.ldw, (size_t)g.Nout, g.K, NCOLS / 2, &maps.w[ws][1]));
  }
  TcGemm gd = g;
  static const char* tl_sel = getenv("PZ_RG_TIMELINE");   // "outproj" | "qk" | "vt" | "p1" | "tail": which launch stamps
  gd.prof = nullptr;
  if (tl_sel) {
    const bool hit = (!strcmp(tl_sel, "outproj") && g.Rb) || (!strcmp(tl_sel, "qk") && g.Nout == 128 && g.K == 256) ||
                     (!strcmp(tl_sel, "vt") && g.YT) || (!strcmp(tl_sel, "p1") && g.K == 64) || (!strcmp(tl_sel, "tail") && g.Ymax);
    if (hit) gd.prof = kernel_timeline_buffer(2048 + 1024);
  }
  PZ_CUDA(launch_pdl(kern, dim3(2 * per * nsets), dim3(RP_THREADS), smem, st, gd, maps));
  PZ_LAUNCH_CHECK();
  return 0;
}

// Row-major split GEMM.  Operands: X / Xlo [M, K] and W / Wlo [Nout, K] fp16 planes (same leading dimensions);
// outputs: Yf fp32 and/or Yb + Yblo fp16 planes and/or YT + YTlo transposed planes and/or Ymax [M / 128, ldmax] = the
// column maxima of every 128-row tile; residual Rf (fp32) or Rb + Rblo.
int launch_split_rowgemm(const TcGemm& g, cudaStream_t st) {
  PZ_REQUIRE(g.W[0] && g.Wlo[0] && g.X && g.Xlo && (g.Yf || g.Yb || g.YT || g.Ymax), PZ_ERR_ARG, "split_rowgemm: null operand");
  PZ_REQUIRE((!g.Yb || g.Yblo) && (!g.YT || (g.YTlo && g.t_rows > 0)) && (!g.Rb || g.Rblo), PZ_ERR_ARG,
             "split_rowgemm: a 16-bit tensor needs both of its planes");
  PZ_REQUIRE(g.epi == 0 && !g.rows, PZ_ERR_ARG, "split_rowgemm: store / tile-max epilogue only");
  PZ_REQUIRE(g.K % 64 == 0 && g.Nout % 128 == 0 && g.ldx % 8 == 0 && g.ldw % 8 == 0, PZ_ERR_UNSUPPORTED,
             "split_rowgemm: needs K %% 64 == 0, Nout %% 128 == 0 and 16-byte aligned rows (K=%d Nout=%d)", g.K, g.Nout);
  PZ_REQUIRE((!g.Yb || (g.ldyb % 8 == 0 && ((uintptr_t)g.Yb & 15) == 0 && ((uintptr_t)g.Yblo & 15) == 0)) &&
                 (!g.Yf || (g.ldyf % 4 == 0 && ((uintptr_t)g.Yf & 15) == 0)) &&
                 (!g.Rb || (g.ldrb % 8 == 0 && ((uintptr_t)g.Rb & 15) == 0 && ((uintptr_t)g.Rblo & 15) == 0)) &&
                 (!g.Rf || (g.ldrf % 4 == 0 && ((uintptr_t)g.Rf & 15) == 0)) &&
                 (!g.rowbias || (g.rb_ld % 4 == 0 && ((uintptr_t)g.rowbias & 15) == 0)),
             PZ_ERR_ARG, "split_rowgemm: outputs / residuals / rowbias must have 16-byte aligned rows");
  PZ_REQUIRE((((uintptr_t)g.X | (uintptr_t)g.Xlo | (uintptr_t)g.W[0] | (uintptr_t)g.Wlo[0] | (uintptr_t)g.W[1] |
               (uintptr_t)g.Wlo[1]) & 15) == 0, PZ_ERR_ARG, "split_rowgemm: operands must be 16-byte aligned");
  const int nsets = (g.rows_per_wset > 0 && g.M > g.rows_per_wset) ? 2 : 1;
  if (nsets == 2)
    PZ_REQUIRE(g.W[1] && g.Wlo[1] && g.M == 2 * g.rows_per_wset, PZ_ERR_ARG, "split_rowgemm: two weight sets need M == 2*rows_per_wset");
  PZ_REQUIRE(g.M % (128 * nsets) == 0, PZ_ERR_UNSUPPORTED, "split_rowgemm: M=%d must be a multiple of %d", g.M, 128 * nsets);
  if (g.n_valid > 0) PZ_REQUIRE(g.n_valid % 32 == 0, PZ_ERR_ARG, "split_rowgemm: n_valid must be a multiple of 32");
  if (g.YT) PZ_REQUIRE(g.t_rows % 128 == 0, PZ_ERR_ARG, "split_rowgemm: t_rows must be a multiple of 128");
  // 256-column tiles halve the re-reads of X but leave at most two tiles per CTA at M = 32768 (the epilogue of a tile then
  // has little to overlap with)
  // CTA-pair kernels (cta_group::2) whenever the rows tile by 256 per weight set
  if (g.M % (256 * nsets) == 0) {
    if (g.Nout == 256 && !g.Ymax) {
      if (split_rowgemm_pair_smem(g, 256, 3, true) <= 232448) return split_rowgemm_pair_launch<256, 3, true>(g, st);
      if (split_rowgemm_pair_smem(g, 256, 2, true) <= 232448) return split_rowgemm_pair_launch<256, 2, true>(g, st);
    }
    if (g.Nout == 128 && !g.Ymax) {
      if (split_rowgemm_pair_smem(g, 128, 4, true) <= 232448) return split_rowgemm_pair_launch<128, 4, true>(g, st);
      if (split_rowgemm_pair_smem(g, 128, 2, true) <= 232448) return split_rowgemm_pair_launch<128, 2, true>(g, st);
    }
    if (g.Nout % 256 == 0) {
      if (split_rowgemm_pair_smem(g, 256, 3, false) <= 232448) return split_rowgemm_pair_launch<256, 3, false>(g, st);
      return split_rowgemm_pair_launch<256, 2, false>(g, st);
    }
  }
  // the one-CTA kernels: rows that tile only by 128 per weight set (pz_group_mlp_maxpool with B*N = 128 mod 256), and
  // 128-column outputs with a tile-max epilogue
  if (g.Nout % 256 == 0) return split_rowgemm_launch<256, 2>(g, st);
  return split_rowgemm_launch<128, 3>(g, st);
}

// 16-byte read-only global load as a VOLATILE asm: ptxas moves plain __ldg loads freely -- in the gather producers it
// sank the loads of the next half-stage behind the stores of the current one (SASS: all 16 LDG.128 of a job issued back
// to back right before the barrier arrival), so nothing was in flight while the operand was formed and every job began
// with a full L2 latency (50 % of the producers' samples).  Volatile asm statements keep their program order relative to
// the (volatile) st.shared of the operand.
__device__ __forceinline__ float4 ldg_nc_pinned(const float4* p) {
  float4 v;
  asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}

// ============================================================================================== gathered GEMM
//   D^T[ch, r] = sum_k W[ch, k] * relu(P[rows[r], k] - Q[r / 32, k])     P [*, K] and Q [M / 32, K] fp32 (Q[g, k] =
//   W1x[k, 0:3] . centre_g, written by centre_proj_f32_kernel)
// channels on UMMA M (TMEM lanes), the ROWS gathered rows of a tile on UMMA N (TMEM columns): the max over the 32
// neighbours of a group is an in-thread reduction over 32 consecutive columns.  One 128-channel block per CTA (the
// CTAs of a weight set are split between the channel blocks), both planes of its weights resident in shared memory.
// Producers (8 warps): P rows are fp32 in global memory; they are loaded one half-stage ahead into registers (fully
// coalesced LDG.128, the row ids one TILE ahead), relu(P - Q) is formed in fp32, split into hi / lo and each plane is
// written with one swizzled st.shared -- the operand is written once and never re-read by the producers.
// (16 producer warps, twice the warps per scheduler to hide the latencies of the producer chain, measured slower: 0.242 vs
// 0.229 ms)
template <int ROWS, int NST>
__global__ void __launch_bounds__(SG_THREADS, 1) split_gather_kernel(const TcGemm g) {
  extern __shared__ __align__(1024) uint8_t sgg_smem_raw[];
  const uint32_t smem_base = (smem_u32(sgg_smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = sgg_smem_raw + (smem_base - smem_u32(sgg_smem_raw));
  constexpr int EPI = 4, PW = 8, PROD_THREADS = PW * 32, THREADS = SG_THREADS, RP = PW * 4;   // RP: rows per producer pass
  constexpr uint32_t X_PLANE = ROWS * 128, STAGE = 2 * X_PLANE;
  const int kblocks = g.K / KB;
  const uint32_t w_plane = (uint32_t)kblocks * TILE16K;          // resident: [W hi kblocks tiles][W lo kblocks tiles]
  const uint32_t stages_base = smem_base + 2 * w_plane;
  const uint32_t bars = stages_base + NST * STAGE;
  const uint32_t full_bar = bars, empty_bar = bars + 8 * NST, accf_bar = bars + 16 * NST, acce_bar = accf_bar + 16;
  const uint32_t tmem_slot = acce_bar + 16;
  const uint32_t qring_s = tmem_slot + 16;                       // 2 x [ROWS/32 groups][64 ch] fp32 Q tiles (16-byte aligned)

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // partitions: (weight set, 128-channel block); the CTAs are split evenly between them
  const int nsets = (g.rows_per_wset > 0 && g.M > g.rows_per_wset) ? 2 : 1;
  const int chblocks = g.Nout / 128, nparts = nsets * chblocks;
  const int row_tiles = g.M / ROWS, tiles_per_set = row_tiles / nsets;
  const int ctas_per_part = gridDim.x / nparts;
  const int part = min((int)blockIdx.x / ctas_per_part, nparts - 1);
  const int wset = part / chblocks, chb = part - wset * chblocks;
  const int rank = blockIdx.x - part * ctas_per_part;
  const int step = (part == nparts - 1) ? (int)gridDim.x - part * ctas_per_part : ctas_per_part;
  const int tile_begin = wset * tiles_per_set, tile_end = tile_begin + tiles_per_set;
  const __half* __restrict__ Whi = reinterpret_cast<const __half*>(g.W[wset]) + (size_t)chb * 128 * g.ldw;
  const __half* __restrict__ Wlo = reinterpret_cast<const __half*>(g.Wlo[wset]) + (size_t)chb * 128 * g.ldw;
  const float* __restrict__ bias = g.bias[wset];

  if (tid == 0) {
    for (int s = 0; s < NST; ++s) {
      mbar_init(full_bar + 8 * s, PROD_THREADS);
      mbar_init(empty_bar + 8 * s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(accf_bar + 8 * b, 1);
      mbar_init(acce_bar + 8 * b, EPI * 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == EPI) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  {  // resident weights of this channel block: both planes, swizzled [128 ch x 64 k] tiles per k-block
    const int chunks = kblocks * 128 * 8;
    for (int id = tid; id < chunks; id += THREADS) {
      const int c = id & 7, r = (id >> 3) & 127, kb = id >> 10;
      const size_t off = (size_t)r * g.ldw + kb * KB + c * 8;
      *reinterpret_cast<uint4*>(smem_gen + (size_t)kb * TILE16K + sw128(r, c)) = *reinterpret_cast<const uint4*>(Whi + off);
      *reinterpret_cast<uint4*>(smem_gen + w_plane + (size_t)kb * TILE16K + sw128(r, c)) = *reinterpret_cast<const uint4*>(Wlo + off);
    }
    fence_proxy_async();
  }
  // the weight planes above were packed at least two launches ago (complete before this grid can be resident, see pdl_enter)
  pdl_enter();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  if (warp > EPI) {
    // =========================================================== producers
    constexpr int CH = ROWS / RP;                 // chunks per thread per stage (rows r0 + RP i)
    constexpr int QV = (ROWS / 32) * 16;          // float4 pieces of one stage's Q tile ([groups][64 ch] fp32)
    const int pt = tid - (EPI + 1) * 32, gc = pt & 7, r0 = pt >> 3;
    int my_tiles = 0;
    for (int t = tile_begin + rank; t < tile_end; t += step) ++my_tiles;
    const int jobs = my_tiles * kblocks;          // job j = (tile j / kblocks, k-block j % kblocks)
    const float* __restrict__ P = g.Xf;
    const float* __restrict__ Q = g.Qf;
    // Two half-stages of HC chunks are in flight: the loads of half h of the NEXT job are issued right after half h of
    // this job has been stored.  The loads stay under `if (more)`: the branch keeps ptxas from sinking them behind the
    // barrier arrival (measured: with unconditional loads it groups all of a stage's loads after the arrival and the two
    // halves are no longer staggered, +25 % run time).  A deeper ring (4 units in flight) is SLOWER as well: the kernel
    // is bound by the LSU data pipe (fp32 P in + both operand planes out = 8 bytes per element through a 64 B/clk path;
    // ncu l1tex__data_pipe_lsu_wavefronts 77 %), not by load latency.
    constexpr int HC = CH / 2;
    float4 buf[2][HC][2];
    int ids[CH], ids_n[CH];                       // source rows of the current / the next tile
    // Q tiles go through a two-slot shared-memory ring: thread t < QV fetches ONE float4 of the tile of job j + 2 at
    // the end of job j, parks it in a register for a whole stage, writes it to the ring at the end of job j + 1 (one
    // producer-only barrier per stage); the subtraction then reads Q with LDS broadcasts instead of waiting for L2
    float4 qpre = make_float4(0.f, 0.f, 0.f, 0.f);
    auto q_fetch = [&](int jt) {
      const int ti = jt / kblocks, kb = jt - ti * kblocks;
      const int group0 = ((tile_begin + rank + ti * step) * ROWS) >> 5;
      if (pt < QV) qpre = __ldg(reinterpret_cast<const float4*>(Q + (size_t)(group0 + (pt >> 4)) * g.K + kb * KB + (pt & 15) * 4));
    };
    auto q_commit = [&](int slot) {
      if (pt < QV)
        asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(qring_s + slot * (QV * 16) + pt * 16), "f"(qpre.x), "f"(qpre.y),
                     "f"(qpre.z), "f"(qpre.w) : "memory");
    };
    auto fetch_ids = [&](int ti, int (&dst)[CH]) {
      const int row0 = (tile_begin + rank + ti * step) * ROWS;
#pragma unroll
      for (int i = 0; i < CH; ++i) dst[i] = g.rows[row0 + r0 + RP * i];
    };
    // loads of half h (chunks h*HC .. h*HC+HC-1) of k-block kb, rows taken from the current or the next tile's ids
    auto load_half = [&](int h, int kb, bool next_tile) {
#pragma unroll
      for (int i = 0; i < HC; ++i) {
        const int id = next_tile ? ids_n[h * HC + i] : ids[h * HC + i];
        // piece gc and piece 8 + gc of the row's sixteen 16-byte pieces: the eight lanes of a row read 128 contiguous
        // bytes per instruction (whole sectors; with pieces 2 gc, 2 gc + 1 every sector was fetched by two instructions)
        const float4* src = reinterpret_cast<const float4*>(P + (size_t)id * g.ldx + kb * KB) + gc;
        buf[h][i][0] = ldg_nc_pinned(src);
        buf[h][i][1] = ldg_nc_pinned(src + 8);
      }
    };
    auto store_half = [&](int h, int slot, uint32_t st_addr) {
#pragma unroll
      for (int i = 0; i < HC; ++i) {
        const int ci = h * HC + i, r = r0 + RP * ci;
        float4 q0, q1;   // channels 4 gc .. + 3 and 32 + 4 gc .. + 3
        const uint32_t qa = qring_s + slot * (QV * 16) + (r >> 5) * 256 + gc * 16;
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(q0.x), "=f"(q0.y), "=f"(q0.z), "=f"(q0.w) : "r"(qa));
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(q1.x), "=f"(q1.y), "=f"(q1.z), "=f"(q1.w) : "r"(qa + 128));
        const float4 p0 = buf[h][i][0], p1 = buf[h][i][1];
        uint2 h0, l0, h1, l1;
        split2(fmaxf(p0.x - q0.x, 0.f), fmaxf(p0.y - q0.y, 0.f), h0.x, l0.x);
        split2(fmaxf(p0.z - q0.z, 0.f), fmaxf(p0.w - q0.w, 0.f), h0.y, l0.y);
        split2(fmaxf(p1.x - q1.x, 0.f), fmaxf(p1.y - q1.y, 0.f), h1.x, l1.x);
        split2(fmaxf(p1.z - q1.z, 0.f), fmaxf(p1.w - q1.w, 0.f), h1.y, l1.y);
        // 4 channels = 8 bytes: half (gc & 1) of 16-byte chunk gc >> 1 (and of chunk 4 + (gc >> 1)) of the swizzled row
        const uint32_t o0 = sw128(r, gc >> 1) + ((gc & 1) << 3), o1 = sw128(r, 4 + (gc >> 1)) + ((gc & 1) << 3);
        asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(st_addr + o0), "r"(h0.x), "r"(h0.y) : "memory");
        asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(st_addr + o1), "r"(h1.x), "r"(h1.y) : "memory");
        asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(st_addr + X_PLANE + o0), "r"(l0.x), "r"(l0.y) : "memory");
        asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(st_addr + X_PLANE + o1), "r"(l1.x), "r"(l1.y) : "memory");
      }
    };
    if (jobs > 0) {
      fetch_ids(0, ids);
      if (my_tiles > 1) fetch_ids(1, ids_n);
      load_half(0, 0, false);
      load_half(1, 0, false);
      q_fetch(0);
      q_commit(0);
      asm volatile("bar.sync 2, %0;" ::"n"(PROD_THREADS) : "memory");
      if (jobs > 1) q_fetch(1);
    }
    for (int j = 0; j < jobs; ++j) {
      const int ti = j / kblocks, kb = j - ti * kblocks;
      const uint32_t s = (uint32_t)j % NST, ph = ((uint32_t)j / NST) & 1;
      const uint32_t st_addr = stages_base + s * STAGE;
      const bool more = j + 1 < jobs;
      const int nkb = (kb + 1 == kblocks) ? 0 : kb + 1;
      const bool new_tile = more && nkb == 0;     // the next job starts the next tile: its rows are ids_n
      mbar_wait(empty_bar + 8 * s, ph ^ 1);
      store_half(0, j & 1, st_addr);
      if (more) load_half(0, nkb, new_tile);      // the registers of half 0 are free again: next job's half 0
      __syncwarp();                               // scheduling fence: ptxas must not sink those loads behind half 1
      store_half(1, j & 1, st_addr);
      fence_proxy_async();
      mbar_arrive(full_bar + 8 * s);
      if (more) load_half(1, nkb, new_tile);
      if (new_tile) {
#pragma unroll
        for (int i = 0; i < CH; ++i) ids[i] = ids_n[i];
        if (ti + 2 < my_tiles) fetch_ids(ti + 2, ids_n);   // needed one whole tile from now
      }
      if (more) {
        q_commit((j + 1) & 1);                    // the tile of job j + 1 (fetched one stage ago) -> its ring slot
        asm volatile("bar.sync 2, %0;" ::"n"(PROD_THREADS) : "memory");
        if (j + 2 < jobs) q_fetch(j + 2);
      }
    }
  } else if (warp == EPI) {
    // =========================================================== MMA issuer (one thread)
    if (lane == 0) {
      const uint32_t idesc = make_idesc_f16(ROWS);
      uint32_t it = 0, tcn = 0;
      for (int t = tile_begin + rank; t < tile_end; t += step, ++tcn) {
        const uint32_t buf = tcn & 1, aph = (tcn >> 1) & 1;
        mbar_wait(acce_bar + 8 * buf, aph ^ 1);
        tc_fence_after();
        for (int kb = 0; kb < kblocks; ++kb, ++it) {
          const uint32_t s = it % NST, ph = (it / NST) & 1;
          mbar_wait(full_bar + 8 * s, ph);
          tc_fence_after();
          const uint32_t st_addr = stages_base + s * STAGE;
          const uint64_t a_hi = make_desc(smem_base + (uint32_t)kb * TILE16K), a_lo = make_desc(smem_base + w_plane + (uint32_t)kb * TILE16K);
          const uint64_t b_hi = make_desc(st_addr), b_lo = make_desc(st_addr + X_PLANE);
#pragma unroll
          for (int k4 = 0; k4 < KB / 16; ++k4)
            umma_split(tmem_base + buf * ROWS, a_hi + 2 * k4, a_lo + 2 * k4, b_hi + 2 * k4, b_lo + 2 * k4, idesc, (kb | k4) != 0);
          umma_commit(empty_bar + 8 * s);
        }
        umma_commit(accf_bar + 8 * buf);
      }
    }
  } else {
    // =========================================================== epilogue: thread = channel, max over groups of 32 rows
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
    const int ch = chb * 128 + warp * 32 + lane;
    const float bv = bias ? bias[ch] : 0.f;
    __half* Ybhi = reinterpret_cast<__half*>(g.Yb);
    __half* Yblo = reinterpret_cast<__half*>(g.Yblo);
    uint32_t tcn = 0;
    for (int t = tile_begin + rank; t < tile_end; t += step, ++tcn) {
      const int row0 = t * ROWS;
      const uint32_t buf = tcn & 1, aph = (tcn >> 1) & 1;
      mbar_wait(accf_bar + 8 * buf, aph);
      tc_fence_after();
      const uint32_t t_addr = tmem_base + lane_base + buf * ROWS;
#pragma unroll 1
      for (int c32 = 0; c32 < ROWS / 32; ++c32) {   // one group of 32 neighbours per TMEM load
        float v[32];
        tmem_ld32(t_addr + c32 * 32, v);
#pragma unroll
        for (int w = 32; w >= 2; w >>= 1) {
#pragma unroll
          for (int i = 0; i < w / 2; ++i) v[i] = fmaxf(v[i], v[i + w / 2]);
        }
        float x = v[0] + bv;
        if (g.relu) x = fmaxf(x, 0.f);
        const size_t grow = (size_t)(row0 >> 5) + c32;
        if (g.Yf) g.Yf[grow * g.ldyf + ch] = x;
        if (Ybhi) {
          const __half hi = __float2half_rn(x);
          Ybhi[grow * g.ldyb + ch] = hi;
          Yblo[grow * g.ldyb + ch] = __float2half_rn(x - __half2float(hi));
        }
      }
      tc_fence_before();
      mbar_arrive(acce_bar + 8 * buf);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == EPI) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------- CTA-pair variant
// Nout == 256: the two CTAs of a cluster (the two SMs of a TPC) hold one 128-channel block of the weights each and
// execute ONE tcgen05.mma.cta_group::2 of M = 256 channels x N = 256 gathered rows per K step.  The B operand of such
// an MMA is split between the pair -- each CTA forms relu(P - Q) for 128 of the 256 rows, in its own shared memory at
// the same offset -- so every gathered row is fetched, transformed and written ONCE for all 256 channels (the
// one-CTA kernel above makes two passes, one per channel block), and each SM reads half the operand bytes per MMA flop.
// Protocol: the leader (cluster rank 0) owns the full / accumulator-empty barriers (one arrival per producer / epilogue
// warp of BOTH CTAs, remote arrivals through mapa); the stage-empty and accumulator-full barriers exist in both CTAs and
// are signalled by multicast tcgen05.commit.
template <int NST>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(SG_THREADS, 1) split_gather_pair_kernel(const TcGemm g) {
  extern __shared__ __align__(1024) uint8_t sgp_smem_raw[];
  // three stages + 128 KB of weights leave no room for an alignment pad: the dynamic shared memory of a kernel without
  // static shared memory starts 1024-aligned; anything else must fail loudly
  const uint32_t smem_base = smem_u32(sgp_smem_raw);
  if ((smem_base & 1023u) != 0) __trap();
  uint8_t* smem_gen = sgp_smem_raw;
  constexpr int EPI = 4, PROD_THREADS = 256, ROWS = 128, NPAIR = 2 * ROWS;
  constexpr uint32_t X_PLANE = ROWS * 128, STAGE = 2 * X_PLANE;
  const int kblocks = g.K / KB;
  const uint32_t w_plane = (uint32_t)kblocks * TILE16K;
  const uint32_t stages_base = smem_base + 2 * w_plane;
  const uint32_t bars = stages_base + NST * STAGE;
  const uint32_t full_bar = bars, empty_bar = bars + 8 * NST, accf_bar = bars + 16 * NST, acce_bar = accf_bar + 16;
  const uint32_t pfull_bar = acce_bar + 16;                      // leader only: stage s of the PEER is full
  const uint32_t tmem_slot = pfull_bar + 8 * NST;
  const uint32_t qring_s = (tmem_slot + 16 + 15) & ~15u;         // 2 x [4 groups][64 ch] fp32 Q tiles

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t crank = cluster_ctarank();
  const int npairs = gridDim.x >> 1, pair = blockIdx.x >> 1;
  const int nsets = (g.rows_per_wset > 0 && g.M > g.rows_per_wset) ? 2 : 1;
  const int pairs_per_set = npairs / nsets;
  const int wset = min(pair / pairs_per_set, nsets - 1);
  const int rank = pair - wset * pairs_per_set;
  const int step = (wset == nsets - 1) ? npairs - wset * pairs_per_set : pairs_per_set;
  const int tiles_per_set = g.M / NPAIR / nsets;
  const int tile_begin = wset * tiles_per_set, tile_end = tile_begin + tiles_per_set;
  const __half* __restrict__ Whi = reinterpret_cast<const __half*>(g.W[wset]) + (size_t)crank * 128 * g.ldw;
  const __half* __restrict__ Wlo = reinterpret_cast<const __half*>(g.Wlo[wset]) + (size_t)crank * 128 * g.ldw;
  const float* __restrict__ bias = g.bias[wset];

  if (tid == 0) {
    for (int s = 0; s < NST; ++s) {
      mbar_init(full_bar + 8 * s, PROD_THREADS);
      mbar_init(empty_bar + 8 * s, 1);
      mbar_init(pfull_bar + 8 * s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(accf_bar + 8 * b, 1);
      mbar_init(acce_bar + 8 * b, 2 * EPI);          // used in the leader only
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == EPI) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  {  // resident weights of this CTA's channel block: both planes, swizzled [128 ch x 64 k] tiles per k-block
    const int chunks = kblocks * 128 * 8;
    for (int id = tid; id < chunks; id += SG_THREADS) {
      const int c = id & 7, r = (id >> 3) & 127, kb = id >> 10;
      const size_t off = (size_t)r * g.ldw + kb * KB + c * 8;
      *reinterpret_cast<uint4*>(smem_gen + (size_t)kb * TILE16K + sw128(r, c)) = *reinterpret_cast<const uint4*>(Whi + off);
      *reinterpret_cast<uint4*>(smem_gen + w_plane + (size_t)kb * TILE16K + sw128(r, c)) = *reinterpret_cast<const uint4*>(Wlo + off);
    }
    fence_proxy_async();
  }
  // the weight planes above were packed at least two launches ago (complete before this grid can be resident, see pdl_enter)
  pdl_enter();
  tc_fence_before();
  cluster_sync_all();        // barriers initialised, TMEM allocated and weights resident in BOTH CTAs
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  if (warp > EPI) {
    // =========================================================== producers (both CTAs): 128 of the 256 rows each
    constexpr int CH = ROWS / 32, HC = CH / 2, QV = (ROWS / 32) * 16;
    const int pt = tid - (EPI + 1) * 32, gc = pt & 7, r0 = pt >> 3;
    int my_tiles = 0;
    for (int t = tile_begin + rank; t < tile_end; t += step) ++my_tiles;
    const int jobs = my_tiles * kblocks;
    const float* __restrict__ P = g.Xf;
    const float* __restrict__ Q = g.Qf;
    float4 buf[2][HC][2];
    int ids[CH], ids_n[CH];
    float4 qpre = make_float4(0.f, 0.f, 0.f, 0.f);
    auto tile_row0 = [&](int ti) { return (tile_begin + rank + ti * step) * NPAIR + (int)crank * ROWS; };
    auto q_fetch = [&](int jt) {
      const int ti = jt / kblocks, kb = jt - ti * kblocks;
      const int group0 = tile_row0(ti) >> 5;
      if (pt < QV) qpre = __ldg(reinterpret_cast<const float4*>(Q + (size_t)(group0 + (pt >> 4)) * g.K + kb * KB + (pt & 15) * 4));
    };
    // Q tile layout in the ring: per group 256 B = [first float4 of the 8 channel octets][second float4 of the 8 octets],
    // so that the 8 distinct addresses of a warp's LDS.128 are 128 contiguous bytes (one wavefront, no bank conflict)
    auto q_commit = [&](int slot) {
      if (pt < QV)
        asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(qring_s + slot * (QV * 16) + (pt >> 4) * 256 + (pt & 1) * 128 + ((pt & 15) >> 1) * 16),
                     "f"(qpre.x), "f"(qpre.y), "f"(qpre.z), "f"(qpre.w) : "memory");
    };
    auto fetch_ids = [&](int ti, int (&dst)[CH]) {
      const int row0 = tile_row0(ti);
#pragma unroll
      for (int i = 0; i < CH; ++i) dst[i] = g.rows[row0 + r0 + 32 * i];
    };
    auto load_half = [&](int h, int kb, bool next_tile) {
#pragma unroll
      for (int i = 0; i < HC; ++i) {
        const int id = next_tile ? ids_n[h * HC + i] : ids[h * HC + i];
        const float4* src = reinterpret_cast<const float4*>(P + (size_t)id * g.ldx + kb * KB + gc * 8);
        buf[h][i][0] = ldg_nc_pinned(src);
        buf[h][i][1] = ldg_nc_pinned(src + 1);
      }
    };
    auto store_half = [&](int h, int slot, uint32_t st_addr) {
#pragma unroll
      for (int i = 0; i < HC; ++i) {
        const int ci = h * HC + i, r = r0 + 32 * ci;
        float4 q0, q1;
        const uint32_t qa = qring_s + slot * (QV * 16) + ci * 256 + gc * 16;
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(q0.x), "=f"(q0.y), "=f"(q0.z), "=f"(q0.w) : "r"(qa));
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(q1.x), "=f"(q1.y), "=f"(q1.z), "=f"(q1.w) : "r"(qa + 128));
        const float4 p0 = buf[h][i][0], p1 = buf[h][i][1];
        uint4 oh, ol;
        split2(fmaxf(p0.x - q0.x, 0.f), fmaxf(p0.y - q0.y, 0.f), oh.x, ol.x);
        split2(fmaxf(p0.z - q0.z, 0.f), fmaxf(p0.w - q0.w, 0.f), oh.y, ol.y);
        split2(fmaxf(p1.x - q1.x, 0.f), fmaxf(p1.y - q1.y, 0.f), oh.z, ol.z);
        split2(fmaxf(p1.z - q1.z, 0.f), fmaxf(p1.w - q1.w, 0.f), oh.w, ol.w);
        const uint32_t off = sw128(r, gc);
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(st_addr + off), "r"(oh.x), "r"(oh.y), "r"(oh.z), "r"(oh.w) : "memory");
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(st_addr + X_PLANE + off), "r"(ol.x), "r"(ol.y), "r"(ol.z), "r"(ol.w) : "memory");
      }
    };
    if (jobs > 0) {
      fetch_ids(0, ids);
      if (my_tiles > 1) fetch_ids(1, ids_n);
      load_half(0, 0, false);
      load_half(1, 0, false);
      q_fetch(0);
      q_commit(0);
      asm volatile("bar.sync 2, 256;" ::: "memory");
      if (jobs > 1) q_fetch(1);
    }
    for (int j = 0; j < jobs; ++j) {
      const int ti = j / kblocks, kb = j - ti * kblocks;
      const uint32_t s = (uint32_t)j % NST, ph = ((uint32_t)j / NST) & 1;
      const uint32_t st_addr = stages_base + s * STAGE;
      const bool more = j + 1 < jobs;
      const int nkb = (kb + 1 == kblocks) ? 0 : kb + 1;
      const bool new_tile = more && nkb == 0;
      mbar_wait(empty_bar + 8 * s, ph ^ 1);
      store_half(0, j & 1, st_addr);
      if (more) load_half(0, nkb, new_tile);      // (a scheduling fence here, as in split_gather_kernel, measured slower: 0.294 vs 0.281 ms)
      store_half(1, j & 1, st_addr);
      fence_proxy_async();
      mbar_arrive(full_bar + 8 * s);
      if (more) load_half(1, nkb, new_tile);
      if (new_tile) {
#pragma unroll
        for (int i = 0; i < CH; ++i) ids[i] = ids_n[i];
        if (ti + 2 < my_tiles) fetch_ids(ti + 2, ids_n);
      }
      if (more) {
        q_commit((j + 1) & 1);
        asm volatile("bar.sync 2, 256;" ::: "memory");
        if (j + 2 < jobs) q_fetch(j + 2);
      }
    }
  } else if (warp == EPI) {
    // =========================================================== MMA issuer: one thread of the LEADER CTA
    if (crank == 0 && lane == 0) {
      const uint32_t idesc = make_idesc_f16(NPAIR, 256);
      uint32_t it = 0, tcn = 0;
      for (int t = tile_begin + rank; t < tile_end; t += step, ++tcn) {
        const uint32_t buf = tcn & 1, aph = (tcn >> 1) & 1;
        mbar_wait_cluster(acce_bar + 8 * buf, aph ^ 1);
        tc_fence_after();
        for (int kb = 0; kb < kblocks; ++kb, ++it) {
          const uint32_t s = it % NST, ph = (it / NST) & 1;
          mbar_wait(full_bar + 8 * s, ph);
          mbar_wait_cluster(pfull_bar + 8 * s, ph);
          tc_fence_after();
          const uint32_t st_addr = stages_base + s * STAGE;
          const uint64_t a_hi = make_desc(smem_base + (uint32_t)kb * TILE16K), a_lo = make_desc(smem_base + w_plane + (uint32_t)kb * TILE16K);
          const uint64_t b_hi = make_desc(st_addr), b_lo = make_desc(st_addr + X_PLANE);
#pragma unroll
          for (int k4 = 0; k4 < KB / 16; ++k4) {
            const uint32_t d = tmem_base + buf * NPAIR;
            umma_f16_pair(d, a_hi + 2 * k4, b_hi + 2 * k4, idesc, (kb | k4) != 0);
            umma_f16_pair(d, a_hi + 2 * k4, b_lo + 2 * k4, idesc, 1);
            umma_f16_pair(d, a_lo + 2 * k4, b_hi + 2 * k4, idesc, 1);
          }
          umma_commit_pair(empty_bar + 8 * s);
        }
        umma_commit_pair(accf_bar + 8 * buf);
      }
    } else if (crank == 1 && lane == 0) {
      // relay of the peer CTA: stage s of this CTA is full -> one arrival on the leader's peer-full barrier
      const uint32_t pfull_remote = mapa_shared(pfull_bar, 0);
      int my_tiles = 0;
      for (int t = tile_begin + rank; t < tile_end; t += step) ++my_tiles;
      const uint32_t jobs = (uint32_t)(my_tiles * kblocks);
      for (uint32_t it = 0; it < jobs; ++it) {
        const uint32_t s = it % NST, ph = (it / NST) & 1;
        mbar_wait(full_bar + 8 * s, ph);
        mbar_arrive_cluster(pfull_remote + 8 * s);
      }
    }
  } else {
    // =========================================================== epilogue (both CTAs): thread = channel of this CTA's
    // block, max over the 8 groups of 32 rows of the pair tile
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
    const int ch = (int)crank * 128 + warp * 32 + lane;
    const float bv = bias ? bias[ch] : 0.f;
    __half* Ybhi = reinterpret_cast<__half*>(g.Yb);
    __half* Yblo = reinterpret_cast<__half*>(g.Yblo);
    const uint32_t acce_remote = mapa_shared(acce_bar, 0);
    uint32_t tcn = 0;
    for (int t = tile_begin + rank; t < tile_end; t += step, ++tcn) {
      const int row0 = t * NPAIR;
      const uint32_t buf = tcn & 1, aph = (tcn >> 1) & 1;
      mbar_wait(accf_bar + 8 * buf, aph);
      tc_fence_after();
      const uint32_t t_addr = tmem_base + lane_base + buf * NPAIR;
#pragma unroll 1
      for (int c32 = 0; c32 < NPAIR / 32; ++c32) {   // one group of 32 neighbours per TMEM load
        float v[32];
        tmem_ld32(t_addr + c32 * 32, v);
#pragma unroll
        for (int w = 32; w >= 2; w >>= 1) {
#pragma unroll
          for (int i = 0; i < w / 2; ++i) v[i] = fmaxf(v[i], v[i + w / 2]);
        }
        float x = v[0] + bv;
        if (g.relu) x = fmaxf(x, 0.f);
        const size_t grow = (size_t)(row0 >> 5) + c32;
        if (g.Yf) g.Yf[grow * g.ldyf + ch] = x;
        if (Ybhi) {
          const __half hi = __float2half_rn(x);
          Ybhi[grow * g.ldyb + ch] = hi;
          Yblo[grow * g.ldyb + ch] = __float2half_rn(x - __half2float(hi));
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(acce_remote + 8 * buf);
    }
  }
  tc_fence_before();
  cluster_sync_all();        // the leader's MMAs read the peer's shared memory: nobody leaves before everybody is done
  if (warp == EPI) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

static int split_gather_pair_launch(const TcGemm& g, cudaStream_t st) {
  constexpr int NST = 3;
  const int kblocks = g.K / KB;
  const size_t smem = 2 * (size_t)kblocks * TILE16K + (size_t)NST * 2 * 128 * 128 + 8 * (3 * NST + 4) + 32 +
                      2 * (size_t)4 * 64 * sizeof(float);
  PZ_REQUIRE(smem <= 232448, PZ_ERR_UNSUPPORTED, "split_gather (pair): needs %zu B of shared memory (K=%d)", smem, g.K);
  auto kern = split_gather_pair_kernel<NST>;
  PZ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int nsets = (g.rows_per_wset > 0 && g.M > g.rows_per_wset) ? 2 : 1;
  const int tiles_per_set = g.M / 256 / nsets;
  int per = (kNumSMs / 2) / nsets;                 // CTA pairs per weight set
  if (per > tiles_per_set) per = tiles_per_set;
  if (per < 1) per = 1;
  PZ_CUDA(launch_pdl(kern, dim3(2 * per * nsets), dim3(SG_THREADS), smem, st, g));
  PZ_LAUNCH_CHECK();
  return 0;
}

template <int ROWS, int NST>
static int split_gather_launch(const TcGemm& g, cudaStream_t st) {
  const int kblocks = g.K / KB;
  const size_t smem = 1024 + 2 * (size_t)kblocks * TILE16K + (size_t)NST * 2 * ROWS * 128 + 8 * (2 * NST + 4) + 32 +
                      2 * (size_t)(ROWS / 32) * 64 * sizeof(float);
  PZ_REQUIRE(smem <= 232448, PZ_ERR_UNSUPPORTED, "split_gather: needs %zu B of shared memory (K=%d)", smem, g.K);
  auto kern = split_gather_kernel<ROWS, NST>;
  PZ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int nsets = (g.rows_per_wset > 0 && g.M > g.rows_per_wset) ? 2 : 1;
  const int nparts = nsets * (g.Nout / 128);
  const int tiles_per_part = g.M / ROWS / nsets;
  int per = kNumSMs / nparts;
  if (per > tiles_per_part) per = tiles_per_part;
  if (per < 1) per = 1;
  PZ_CUDA(launch_pdl(kern, dim3(per * nparts), dim3(SG_THREADS), smem, st, g));
  PZ_LAUNCH_CHECK();
  return 0;
}

// gathered split GEMM: Xf = P [*, K] fp32 (ldx), Qf [M/32, K] fp32, rows [M] as in the bf16 gather GEMM, W + Wlo fp16
// planes [Nout, K]; outputs Yf [M/32, ldyf] fp32 and/or Yb + Yblo fp16 planes
int launch_split_gather(const TcGemm& g, cudaStream_t st) {
  PZ_REQUIRE(g.Xf && g.Qf && g.rows && g.W[0] && g.Wlo[0] && (g.Yf || g.Yb), PZ_ERR_ARG, "split_gather: null operand");
  PZ_REQUIRE(((uintptr_t)g.Qf & 15) == 0 && g.epi == 1, PZ_ERR_ARG, "split_gather: Q must be 16-byte aligned; group-max epilogue only");
  PZ_REQUIRE(!g.Yb || g.Yblo, PZ_ERR_ARG, "split_gather: a 16-bit output needs both planes");
  PZ_REQUIRE(g.K % 64 == 0 && g.K <= 256 && g.Nout % 128 == 0 && g.ldx % 4 == 0 && g.ldw % 8 == 0 && ((uintptr_t)g.Xf & 15) == 0 &&
                 (((uintptr_t)g.W[0] | (uintptr_t)g.Wlo[0] | (uintptr_t)g.W[1] | (uintptr_t)g.Wlo[1]) & 15) == 0,
             PZ_ERR_UNSUPPORTED, "split_gather: needs K %% 64 == 0, K <= 256, Nout %% 128 == 0 and 16-byte aligned rows (K=%d Nout=%d)", g.K, g.Nout);
  const int nsets = (g.rows_per_wset > 0 && g.M > g.rows_per_wset) ? 2 : 1;
  if (nsets == 2)
    PZ_REQUIRE(g.W[1] && g.Wlo[1] && g.M == 2 * g.rows_per_wset, PZ_ERR_ARG, "split_gather: two weight sets need M == 2*rows_per_wset");
  if (g.K <= 128) {
    PZ_REQUIRE(g.M % (256 * nsets) == 0, PZ_ERR_UNSUPPORTED, "split_gather: M=%d must be a multiple of %d", g.M, 256 * nsets);
    // (128-row stages, three or four deep, measured slower: 0.258 / 0.262 ms)
    return split_gather_launch<256, 2>(g, st);
  }
  PZ_REQUIRE(g.M % (128 * nsets) == 0, PZ_ERR_UNSUPPORTED, "split_gather: M=%d must be a multiple of %d", g.M, 128 * nsets);
  // 256 output channels on rows that tile by 256 per weight set: one CTA pair per tile (cta_group::2), every gathered row
  // formed once for both channel blocks
  if (g.Nout == 256 && g.M % (256 * nsets) == 0) return split_gather_pair_launch(g, st);
  // any other Nout (C1 = 256 with C2 = 128) or rows that tile only by 128: one CTA per 128-row tile and channel block
  return split_gather_launch<128, 2>(g, st);
}

// fp32 [rows, cols] (row stride ldi) -> fp16 hi / lo planes (row stride ldo)
__global__ void __launch_bounds__(256) split_planes_kernel(const float* __restrict__ in, size_t ldi, size_t rows, int cols,
                                                           __half* __restrict__ hi, __half* __restrict__ lo, size_t ldo) {
  const int c4 = cols / 4;
  const size_t total = rows * c4;
  for (size_t e = (size_t)blockIdx.x * 256 + threadIdx.x; e < total; e += (size_t)gridDim.x * 256) {
    const size_t r = e / c4;
    const int c = (int)(e - r * c4) * 4;
    const float4 v = *reinterpret_cast<const float4*>(in + r * ldi + c);
    uint2 oh, ol;
    split2(v.x, v.y, oh.x, ol.x);
    split2(v.z, v.w, oh.y, ol.y);
    *reinterpret_cast<uint2*>(hi + r * ldo + c) = oh;
    *reinterpret_cast<uint2*>(lo + r * ldo + c) = ol;
  }
}

int launch_split_planes(const float* in, size_t ldi, size_t rows, int cols, void* hi, void* lo, size_t ldo, cudaStream_t st) {
  PZ_REQUIRE(in && hi && lo, PZ_ERR_ARG, "split_planes: null pointer");
  PZ_REQUIRE(cols % 4 == 0 && ldi % 4 == 0 && ldo % 4 == 0 && ((uintptr_t)in & 15) == 0 && (((uintptr_t)hi | (uintptr_t)lo) & 7) == 0,
             PZ_ERR_ARG, "split_planes: needs cols %% 4 == 0 and aligned rows");
  const size_t total = rows * (cols / 4);
  if (total == 0) return 0;
  const size_t want = (total + 255) / 256;
  const int blocks = (int)(want < (size_t)kNumSMs * 16 ? want : (size_t)kNumSMs * 16);
  split_planes_kernel<<<blocks, 256, 0, st>>>(in, ldi, rows, cols, static_cast<__half*>(hi), static_cast<__half*>(lo), ldo);
  PZ_LAUNCH_CHECK();
  return 0;
}

}  // namespace pz
