// tcgen05 TF32 GEMM for the training step: C[m,n] (+)= sum_k A(m,k) B(n,k), fp32 in memory, fp32 accumulate in TMEM,
// operands rounded to TF32 (10-bit mantissa) by the tensor core -- the arithmetic stock PyTorch 1.10 (the version
// the reference pins, README.md:30) uses for every nn.Linear on Ampere-or-newer GPUs (allow_tf32 defaulted to on).
//
// Each operand is either K-major (A[m*lda + k]) or MN-major (A[k*lda + m]); both are staged by cp.async straight
// from the fp32 tensors into SWIZZLE_128B shared-memory tiles, no conversion pass:
//   forward   Y  = X W^T     A = X  K-major,   B = W  K-major
//   dgrad     dX = dY W      A = dY K-major,   B = W  MN-major (B(n=k_in, k=n_out) = W[n_out*ld + k_in])
//   wgrad     dW = dY^T X    A = dY MN-major,  B = X  MN-major, K = the row count -> split-K over the persistent grid,
//                            partial tiles added with fp32 atomics into the pre-zeroed gradient buffer
// Structure follows gemm_tc_rows.cu: 4 producer warps, one MMA thread (tcgen05.mma.kind::tf32, M=128, N=128/256,
// K=8 per instruction, 4 per 32-wide k-block), 8 epilogue warps reading the double-buffered TMEM accumulator
// (thread = output row, 32 consecutive columns per tcgen05.ld), persistent grid of <= 148 CTAs.
#include <stdlib.h>

#include "pz_common.cuh"
#include "tc_common.cuh"

namespace pz {

using namespace tc;

namespace {
constexpr int TG_THREADS = 13 * 32;   // 8 epilogue warps, 1 MMA warp, 4 producer warps
constexpr int TG_EPI = 8, TG_PROD_THREADS = 128;
constexpr int TG_ROWS = 128;          // UMMA M
constexpr int TG_KB = 32;             // fp32 elements per k-block = one 128-byte swizzle row

// K-major:  rows of 128 B (32 k), 8-row atoms, SBO = 1024.
// MN-major (32-bit operands only admit SWIZZLE_128B_BASE32B, cute's Layout_MN_SW128_32B_Atom): 128-byte rows hold 32
//           consecutive MN elements of one k; 4 k-rows form a 512-byte atom whose 32-byte chunks are XOR-swizzled
//           with the row index (Swizzle<2,5,2>); k-atoms are SBO = 512 bytes apart, MN blocks of 32 elements
//           LBO = TG_KB*128 bytes apart.
__device__ __forceinline__ uint64_t make_desc_mn(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((TG_KB * 128) >> 4) << 16;         // leading byte offset, bits [16,30)
  d |= (uint64_t)(512 >> 4) << 32;                   // stride byte offset, bits [32,46)
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)1 << 61;                            // SWIZZLE_128B_BASE32B
  return d;
}
// byte offset of 16-byte chunk c (0..7) of k-row r inside an MN-major block: 32-byte chunk index ^ (r & 3)
__device__ __forceinline__ uint32_t sw128_32(int r, int c) {
  return (uint32_t)(r * 128 + ((((c >> 1) ^ (r & 3)) << 5) | ((c & 1) << 4)));
}
// D = f32, A = B = tf32, majors as given, M = 128, N = n
__host__ __device__ constexpr uint32_t make_idesc_tf32(int n, int a_mn, int b_mn) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
}  // namespace

struct Tf32Gemm {
  const float* A; long long lda; int a_mn;
  const float* B; long long ldb; int b_mn;
  float* C; long long ldc;
  int M, N, K;
  int splitk;                 // >= 1; > 1: atomically add partial tiles into C
  int atomic;                 // splitk > 1 was requested: always add (even if the K range ends up unsplit)
  const float* bias;          // [N] or null
  int relu;
  const float* mask;          // zero where mask[m*ldmask + n] <= 0
  long long ldmask;
  int accumulate;             // C += result (splitk == 1)
  int batch;                  // independent problems at A + i*sA, B + i*sB, C / mask + i*sC (streaming mode only)
  long long sA, sB, sC;
};
// BRES (B resident): when all k-blocks of one B column tile fit in shared memory (a weight matrix: NCOLS * K * 4 bytes
// <= 128 KB) every CTA loads them ONCE, keeps one column tile for its whole life and streams only A -- the streaming
// mode re-reads the B tile for every row tile, which makes the 128/256-wide layers L2-bandwidth bound
// (ncu: 384 KB of L2->SM traffic per 128x256 output tile, 2/3 of it weights).

template <int NCOLS, int NST, bool BRES>
__global__ void __launch_bounds__(TG_THREADS, 1) tf32_gemm_kernel(const Tf32Gemm g) {
  extern __shared__ __align__(1024) uint8_t tg_smem_raw[];
  const uint32_t smem_base = (smem_u32(tg_smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = tg_smem_raw + (smem_base - smem_u32(tg_smem_raw));
  constexpr uint32_t STAGE_A = TG_ROWS * 128, STAGE_B = NCOLS * 128, STAGE = BRES ? STAGE_A : STAGE_A + STAGE_B;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int kblocks = g.K / TG_KB;
  const uint32_t bres_base = smem_base + NST * STAGE;                       // BRES: kblocks B tiles of STAGE_B bytes
  const uint32_t bars = bres_base + (BRES ? (uint32_t)kblocks * STAGE_B : 0u);
  const uint32_t full_bar = bars, empty_bar = bars + 8 * NST, accf_bar = bars + 16 * NST, acce_bar = accf_bar + 16;
  const uint32_t tmem_slot = acce_bar + 16, bres_bar = tmem_slot + 8;
  const int kb_per_split = (kblocks + g.splitk - 1) / g.splitk;
  const int nsplit = (kblocks + kb_per_split - 1) / kb_per_split;       // every split is non-empty
  const int row_tiles = g.M / TG_ROWS, col_tiles = g.N / NCOLS;
  // BRES: CTA b owns column tile b % col_tiles (the grid is a multiple of col_tiles) and row tiles b / col_tiles + i * stride
  const int per_batch = row_tiles * col_tiles * nsplit;
  const int work = BRES ? row_tiles : per_batch * g.batch;
  const int w_begin = BRES ? (int)blockIdx.x / col_tiles : (int)blockIdx.x;
  const int w_step = BRES ? (int)gridDim.x / col_tiles : (int)gridDim.x;
  const int my_ct = BRES ? (int)blockIdx.x % col_tiles : 0;

  if (tid == 0) {
    for (int s = 0; s < NST; ++s) {
      mbar_init(full_bar + 8 * s, TG_PROD_THREADS);
      mbar_init(empty_bar + 8 * s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(accf_bar + 8 * b, 1);
      mbar_init(acce_bar + 8 * b, TG_EPI * 32);
    }
    mbar_init(bres_bar, TG_PROD_THREADS);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == TG_EPI) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  // work item -> (row tile, column tile, k range); the split index varies fastest so that the CTAs working on one
  // output tile run at the same time (their atomics meet in L2)
  auto decode = [&](int w, int& rt, int& ct, int& kb0, int& kb1, int& bi) {
    bi = 0;
    if (BRES) {
      rt = w; ct = my_ct; kb0 = 0; kb1 = kblocks;
      return;
    }
    bi = w / per_batch;
    w -= bi * per_batch;
    const int sp = w % nsplit, t = w / nsplit;
    ct = t % col_tiles;
    rt = t / col_tiles;
    kb0 = sp * kb_per_split;
    kb1 = min(kblocks, kb0 + kb_per_split);
  };

  if (warp > TG_EPI) {
    // ================================================= producers
    const int pt = tid - (TG_EPI + 1) * 32;
    uint32_t issued = 0, arrived = 0;
    auto load_b = [&](uint32_t dst, const float* Bp, int col0, long long k0) {
      if (!g.b_mn) {
        for (int id = pt; id < NCOLS * 8; id += TG_PROD_THREADS) {
          const int c = id & 7, r = id >> 3;
          cp_async16(dst + sw128(r, c), Bp + (long long)(col0 + r) * g.ldb + k0 + c * 4);
        }
      } else {
        constexpr int NB = NCOLS / 32;
        for (int id = pt; id < NCOLS * 8; id += TG_PROD_THREADS) {
          const int c = id & 7, j = (id >> 3) % NB, kk = (id >> 3) / NB;
          cp_async16(dst + j * (TG_KB * 128) + sw128_32(kk, c), Bp + (k0 + kk) * g.ldb + col0 + j * 32 + c * 4);
        }
      }
    };
    if (BRES) {
      for (int kb = 0; kb < kblocks; ++kb) load_b(bres_base + kb * STAGE_B, g.B, my_ct * NCOLS, (long long)kb * TG_KB);
      cp_async_commit();
      cp_async_wait<0>();
      fence_proxy_async();
      mbar_arrive(bres_bar);
    }
    for (int w = w_begin; w < work; w += w_step) {
      int rt, ct, kb0, kb1, bi;
      decode(w, rt, ct, kb0, kb1, bi);
      const int row0 = rt * TG_ROWS, col0 = ct * NCOLS;
      const float* Ab = g.A + (long long)bi * g.sA;
      const float* Bb = g.B + (long long)bi * g.sB;
      for (int kb = kb0; kb < kb1; ++kb) {
        const uint32_t s = issued % NST, ph = (issued / NST) & 1;
        mbar_wait(empty_bar + 8 * s, ph ^ 1);
        const uint32_t st_addr = smem_base + s * STAGE;
        const long long k0 = (long long)kb * TG_KB;
        if (!g.a_mn) {
          for (int id = pt; id < TG_ROWS * 8; id += TG_PROD_THREADS) {
            const int c = id & 7, r = id >> 3;
            cp_async16(st_addr + sw128(r, c), Ab + (long long)(row0 + r) * g.lda + k0 + c * 4);
          }
        } else {
          for (int id = pt; id < TG_ROWS * 8; id += TG_PROD_THREADS) {
            const int c = id & 7, j = (id >> 3) & 3, kk = id >> 5;      // 8 chunks x 4 MN blocks x 32 k
            cp_async16(st_addr + j * (TG_KB * 128) + sw128_32(kk, c), Ab + (k0 + kk) * g.lda + row0 + j * 32 + c * 4);
          }
        }
        if (!BRES) load_b(st_addr + STAGE_A, Bb, col0, k0);
        cp_async_commit();
        ++issued;
        // stages whose loads may be outstanding before the oldest is waited for and published; must stay below NST - 1,
        // otherwise "full" is only signalled once the ring is exhausted and the MMA warp starves (measured: -20 %)
        constexpr int INFLIGHT = NST >= 8 ? 5 : 2;
        if (issued - arrived > INFLIGHT) {
          cp_async_wait<INFLIGHT>();
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
  } else if (warp == TG_EPI) {
    // ================================================= MMA issuer
    if (lane == 0) {
      const uint32_t idesc = make_idesc_tf32(NCOLS, g.a_mn, g.b_mn);
      uint32_t it = 0, tcn = 0;
      if (BRES) {
        mbar_wait(bres_bar, 0);
        tc_fence_after();
      }
      for (int w = w_begin; w < work; w += w_step, ++tcn) {
        int rt, ct, kb0, kb1, bi;
        decode(w, rt, ct, kb0, kb1, bi);
        const uint32_t buf = tcn & 1, aph = (tcn >> 1) & 1;
        mbar_wait(acce_bar + 8 * buf, aph ^ 1);
        tc_fence_after();
        for (int kb = kb0; kb < kb1; ++kb, ++it) {
          const uint32_t s = it % NST, ph = (it / NST) & 1;
          mbar_wait(full_bar + 8 * s, ph);
          tc_fence_after();
          const uint32_t st_addr = smem_base + s * STAGE;
          const uint64_t adesc = g.a_mn ? make_desc_mn(st_addr) : make_desc(st_addr);
          const uint32_t b_addr = BRES ? bres_base + (uint32_t)kb * STAGE_B : st_addr + STAGE_A;
          const uint64_t bdesc = g.b_mn ? make_desc_mn(b_addr) : make_desc(b_addr);
          const uint32_t astep = g.a_mn ? (1024 >> 4) : (32 >> 4), bstep = g.b_mn ? (1024 >> 4) : (32 >> 4);
#pragma unroll
          for (int k8 = 0; k8 < TG_KB / 8; ++k8)
            umma_tf32(tmem_base + buf * NCOLS, adesc + astep * k8, bdesc + bstep * k8, idesc, (kb != kb0) || k8 != 0);
          umma_commit(empty_bar + 8 * s);
        }
        umma_commit(accf_bar + 8 * buf);
      }
    }
  } else {
    // ================================================= epilogue: thread = row, 32 columns per TMEM load
    const int quarter = warp & 3, half = warp >> 2;
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    uint32_t tcn = 0;
    for (int w = w_begin; w < work; w += w_step, ++tcn) {
      int rt, ct, kb0, kb1, bi;
      decode(w, rt, ct, kb0, kb1, bi);
      const int col0 = ct * NCOLS;
      const long long row = (long long)rt * TG_ROWS + quarter * 32 + lane;
      float* Cb = g.C + (long long)bi * g.sC;
      const float* maskb = g.mask ? g.mask + (long long)bi * g.sC : nullptr;
      const uint32_t buf = tcn & 1, aph = (tcn >> 1) & 1;
      mbar_wait(accf_bar + 8 * buf, aph);
      tc_fence_after();
#pragma unroll 1
      for (int c32 = half; c32 < NCOLS / 32; c32 += 2) {
        const int cb = col0 + c32 * 32;
        float v[32];
        tmem_ld32(tmem_base + lane_base + buf * NCOLS + c32 * 32, v);
        float* cp = Cb + row * g.ldc + cb;
        if (g.atomic) {
#pragma unroll
          for (int i = 0; i < 32; ++i) atomicAdd(cp + i, v[i]);
          continue;
        }
        if (g.bias) {
#pragma unroll
          for (int q4 = 0; q4 < 8; ++q4) {
            const float4 b4 = *reinterpret_cast<const float4*>(g.bias + cb + q4 * 4);
            v[q4 * 4] += b4.x; v[q4 * 4 + 1] += b4.y; v[q4 * 4 + 2] += b4.z; v[q4 * 4 + 3] += b4.w;
          }
        }
        if (g.accumulate) {
#pragma unroll
          for (int q4 = 0; q4 < 8; ++q4) {
            const float4 b4 = *reinterpret_cast<const float4*>(cp + q4 * 4);
            v[q4 * 4] += b4.x; v[q4 * 4 + 1] += b4.y; v[q4 * 4 + 2] += b4.z; v[q4 * 4 + 3] += b4.w;
          }
        }
        if (g.relu) {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.f);
        }
        if (g.mask) {
          const float* mp = maskb + row * g.ldmask + cb;
#pragma unroll
          for (int q4 = 0; q4 < 8; ++q4) {
            const float4 m4 = *reinterpret_cast<const float4*>(mp + q4 * 4);
            if (!(m4.x > 0.f)) v[q4 * 4] = 0.f;
            if (!(m4.y > 0.f)) v[q4 * 4 + 1] = 0.f;
            if (!(m4.z > 0.f)) v[q4 * 4 + 2] = 0.f;
            if (!(m4.w > 0.f)) v[q4 * 4 + 3] = 0.f;
          }
        }
#pragma unroll
        for (int q4 = 0; q4 < 8; ++q4)
          *reinterpret_cast<float4*>(cp + q4 * 4) = make_float4(v[q4 * 4], v[q4 * 4 + 1], v[q4 * 4 + 2], v[q4 * 4 + 3]);
      }
      tc_fence_before();
      mbar_arrive(acce_bar + 8 * buf);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == TG_EPI) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

template <int NCOLS, int NST, bool BRES>
static int tf32_launch(const Tf32Gemm& g, cudaStream_t st) {
  const int kblocks = g.K / TG_KB;
  const size_t stage = BRES ? (size_t)TG_ROWS * 128 : (size_t)(TG_ROWS * 128 + NCOLS * 128);
  const size_t smem = 1024 + (size_t)NST * stage + (BRES ? (size_t)kblocks * NCOLS * 128 : 0) + 8 * (2 * NST + 6) + 64;
  auto kern = tf32_gemm_kernel<NCOLS, NST, BRES>;
  PZ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int grid;
  if (BRES) {
    const int col_tiles = g.N / NCOLS, row_tiles = g.M / TG_ROWS;
    int per_ct = kNumSMs / col_tiles;                       // CTAs per column tile
    if (per_ct > row_tiles) per_ct = row_tiles;
    grid = per_ct * col_tiles;
  } else {
    const int kbps = (kblocks + g.splitk - 1) / g.splitk;
    const int nsplit = (kblocks + kbps - 1) / kbps;
    const long long work = (long long)(g.M / TG_ROWS) * (g.N / NCOLS) * nsplit * g.batch;
    grid = (int)(work < kNumSMs ? work : kNumSMs);
  }
  kern<<<grid, TG_THREADS, smem, st>>>(g);
  PZ_LAUNCH_CHECK();
  return 0;
}

}  // namespace pz

using namespace pz;

extern "C" int pz_gemm_tf32(int a_mn_major, int b_mn_major, int M, int N, int K, const float* A, long long lda,
                            const float* B, long long ldb, float* C, long long ldc, int splitk,
                            const float* bias_or_null, int relu, const float* mask_or_null, long long ldmask,
                            int accumulate, pz_stream_t stream) {
  return pz_gemm_tf32_batched(a_mn_major, b_mn_major, M, N, K, A, lda, B, ldb, C, ldc, 1, 0, 0, 0, splitk, bias_or_null,
                              relu, mask_or_null, ldmask, accumulate, stream);
}

extern "C" int pz_gemm_tf32_batched(int a_mn_major, int b_mn_major, int M, int N, int K, const float* A, long long lda,
                                    const float* B, long long ldb, float* C, long long ldc, int batch, long long strideA,
                                    long long strideB, long long strideC, int splitk, const float* bias_or_null,
                                    int relu, const float* mask_or_null, long long ldmask, int accumulate,
                                    pz_stream_t stream) {
  PZ_REQUIRE(batch >= 0, PZ_ERR_ARG, "pz_gemm_tf32: batch < 0");
  if (batch == 0) return PZ_OK;
  PZ_REQUIRE(batch == 1 || (splitk == 1 && strideA % 4 == 0 && strideB % 4 == 0 && strideC % 4 == 0), PZ_ERR_ARG,
             "pz_gemm_tf32: batched problems need 16-byte aligned strides and splitk == 1");
  PZ_REQUIRE(M >= 0 && N >= 0 && K >= 0, PZ_ERR_ARG, "pz_gemm_tf32: negative size");
  if (M == 0 || N == 0) return PZ_OK;
  PZ_REQUIRE(A && B && C, PZ_ERR_ARG, "pz_gemm_tf32: null pointer");
  PZ_REQUIRE(M % 128 == 0 && N % 64 == 0 && K % 32 == 0 && K >= 32, PZ_ERR_UNSUPPORTED,
             "pz_gemm_tf32: needs M %% 128 == 0, N %% 64 == 0, K %% 32 == 0 (M=%d N=%d K=%d)", M, N, K);
  PZ_REQUIRE(lda % 4 == 0 && ldb % 4 == 0 && ldc % 4 == 0 && ((uintptr_t)A & 15) == 0 && ((uintptr_t)B & 15) == 0 &&
                 ((uintptr_t)C & 15) == 0,
             PZ_ERR_ARG, "pz_gemm_tf32: operands and output need 16-byte aligned rows");
  PZ_REQUIRE(!bias_or_null || ((uintptr_t)bias_or_null & 15) == 0, PZ_ERR_ARG, "pz_gemm_tf32: bias must be 16-byte aligned");
  PZ_REQUIRE(!mask_or_null || (ldmask % 4 == 0 && ((uintptr_t)mask_or_null & 15) == 0), PZ_ERR_ARG,
             "pz_gemm_tf32: mask needs 16-byte aligned rows");
  PZ_REQUIRE(splitk >= 1, PZ_ERR_ARG, "pz_gemm_tf32: splitk must be >= 1");
  PZ_REQUIRE(!(splitk > 1 && (bias_or_null || relu || mask_or_null || accumulate)), PZ_ERR_UNSUPPORTED,
             "pz_gemm_tf32: split-K adds raw partial sums into a pre-zeroed C (no epilogue)");
  Tf32Gemm g{A, lda, a_mn_major ? 1 : 0, B, ldb, b_mn_major ? 1 : 0, C, ldc, M, N, K, splitk, splitk > 1 ? 1 : 0,
             bias_or_null, relu, mask_or_null, ldmask, accumulate, batch, strideA, strideB, strideC};
  // weights-resident mode: forward / data-gradient GEMMs whose B operand (one 128-column tile, all of K) fits in 128 KB
  // and that have enough row tiles to amortise loading it once per CTA
  // (measured: 17 % faster than streaming for the 128-wide layers, 4.7 TB/s on compulsory bytes; for N = 256 the A
  // operand would be read once per column tile, which costs more than the weights it saves)
  if (batch == 1 && splitk == 1 && N == 128 && M / 128 >= 4 * kNumSMs) {
    if (K <= 128) return tf32_launch<128, 8, true>(g, as_stream(stream));     // 64 KB of weights + 8 x 16 KB of A in flight
    if (K <= 256) return tf32_launch<128, 4, true>(g, as_stream(stream));     // 128 KB + 4 x 16 KB
  }
  if (N % 256 == 0) return tf32_launch<256, 4, false>(g, as_stream(stream));
  if (N % 128 == 0) return tf32_launch<128, 4, false>(g, as_stream(stream));
  return tf32_launch<64, 6, false>(g, as_stream(stream));                     // the 64-wide layers (q, k, stem, heads)
}
