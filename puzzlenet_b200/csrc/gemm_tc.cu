// tcgen05 (5th-gen tensor core) GEMM family for the bf16 path (PZ_PREC_BF16), sm_100a only.
//
//   D^T[ch, row] = sum_k W[ch,k] * X[row,k]          (bf16 x bf16 -> fp32 in TMEM)
//
// The product is computed TRANSPOSED: output channels are the UMMA M dimension (TMEM lanes, one
// per epilogue thread) and activation rows are the UMMA N dimension (TMEM columns).  Both operands
// are K-major in shared memory, which is the natural layout of nn.Linear weights [out,in] and of
// activations [rows,in].  With rows along TMEM columns, the max-pools of the model become purely
// in-thread reductions over consecutive columns:
//   * neighbourhood max-pool over the K=32 rows of a group (model5_b.py:454, :461)
//   * point max-pool over the 256 rows of a cloud            (model5_b.py:475)
// and a plain store writes 32 consecutive channels per warp instruction (coalesced).
//
// Warp roles (13 warps, 1 CTA/SM, persistent over tiles):
//   warps 0-3  epilogue: tcgen05.ld accumulator -> bias/ReLU/residual/max -> global
//   warp  4    TMEM allocation + the single MMA-issuing thread
//   warps 5-12 producers: fill the K-major SWIZZLE_128B operand stages, either with cp.async copies
//              (plain activations / streamed weights) or by *computing* the operand on the fly:
//              grouped-MLP layer 2 gathers  relu(P[rows[r]] - Q[r/32])  (pointnet_util.py:123-130 +
//              model5_b.py:452) so the [B,S,K,3+D] tensor and its layer-1 activations never exist.
// Pipelines: smem stages (full/empty mbarriers, tcgen05.commit frees a stage) and a double-buffered
// TMEM accumulator (accum_full/accum_empty) so the epilogue of tile i overlaps the MMAs of tile i+1.
#include <cuda_bf16.h>

#include "pz_common.cuh"
#include "tc_common.cuh"

namespace pz {

namespace tc {
constexpr int THREADS = 13 * 32;  // 416: epilogue + MMA + producer warps (split depends on the operand mode)
}  // namespace tc

using namespace tc;

__device__ __forceinline__ void tl_stamp(long long* prof, int slot) {
  if (prof != nullptr && blockIdx.x == 0) prof[slot] = clock64();
}

// ROWS: activation rows per tile (UMMA N).  NCHB: 128-channel blocks per tile (accumulators).
// RESIDENT: all of W for the tile's NCHB blocks stays in smem (K*NCHB*256 bytes).  GATHER: computed B.
template <int ROWS, int NCHB, bool RESIDENT, bool GATHER, int NST>
__global__ void __launch_bounds__(THREADS, 1) tc_gemm_kernel(const TcGemm g) {
  extern __shared__ __align__(1024) uint8_t tc_smem_raw[];
  // carve: [resident W][stages][barriers]
  const uint32_t smem_base = (smem_u32(tc_smem_raw) + 1023u) & ~1023u;
  const int kblocks = g.K / KB;
  const uint32_t w_block_bytes = 128 * 128;                     // one [128 ch x 64 k] block
  const uint32_t resident_bytes = RESIDENT ? (uint32_t)(NCHB * kblocks) * w_block_bytes : 0u;
  constexpr uint32_t STAGE_W_BYTES = RESIDENT ? 0u : (uint32_t)NCHB * 128u * 128u;
  constexpr uint32_t STAGE_X_BYTES = (uint32_t)ROWS * 128u;
  constexpr uint32_t STAGE_BYTES = STAGE_W_BYTES + STAGE_X_BYTES;
  const uint32_t stages_base = smem_base + resident_bytes;
  const uint32_t bars_base = stages_base + NST * STAGE_BYTES;   // 8-byte aligned (multiple of 1024)
  const uint32_t full_bar = bars_base, empty_bar = bars_base + 8 * NST;
  const uint32_t accf_bar = bars_base + 16 * NST, acce_bar = accf_bar + 16;
  const uint32_t tmem_slot = acce_bar + 16;
  // GATHER extras (16-byte aligned): NST x [ROWS/32 groups][64] bf16 Q tiles, NST x [ROWS/32][4] fp32 group centres,
  // and the layer-1 xyz weights W1[:,0:3] of all K channels as float4 (resident)
  const uint32_t qstage_base = tmem_slot + 16;
  const uint32_t cstage_base = qstage_base + NST * (ROWS / 32) * 128;
  const uint32_t w1x_base = cstage_base + NST * (ROWS / 32) * 16;
  __shared__ float sxyz[ROWS * 3];
  uint8_t* smem_gen = tc_smem_raw + (smem_base - smem_u32(tc_smem_raw));   // generic pointer to smem_base

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // Role split.  Plain operands (cp.async) need few producer threads but a heavy store epilogue, so two
  // epilogue warps share each TMEM lane quarter (a warp may only touch lanes 32*(warp%4)..+31) and take
  // alternate 32-column chunks; the gather mode computes its operand and keeps 8 producer warps.
  constexpr int EPI_WARPS = GATHER ? 4 : 8, PROD_WARPS = 12 - EPI_WARPS, PROD_THREADS = PROD_WARPS * 32;

  // ---- tile partition: CTAs are split between the weight sets so a CTA never switches weights
  const int nsets = (g.rows_per_wset > 0 && g.M > g.rows_per_wset) ? 2 : 1;
  const int row_tiles = g.M / ROWS;
  const int ch_tiles = g.Nout / (128 * NCHB);
  const int tiles_per_set = (row_tiles / nsets) * ch_tiles;
  const int ctas_per_set = gridDim.x / nsets;
  const int wset = min((int)blockIdx.x / ctas_per_set, nsets - 1);
  const int rank_in_set = blockIdx.x - wset * ctas_per_set;
  const int step = (wset == nsets - 1) ? (int)gridDim.x - wset * ctas_per_set : ctas_per_set;
  const int tile_begin = wset * tiles_per_set;
  const __nv_bfloat16* __restrict__ W = g.W[wset];
  const float* __restrict__ bias = g.bias[wset];

  if (tid == 0) {
    for (int s = 0; s < NST; ++s) {
      mbar_init(full_bar + 8 * s, 128);   // gather: one 128-thread producer group per stage; plain: 4 producer warps
      mbar_init(empty_bar + 8 * s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(accf_bar + 8 * b, 1);
      mbar_init(acce_bar + 8 * b, EPI_WARPS * 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == EPI_WARPS) {  // TMEM allocation by one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (RESIDENT) {  // whole weight matrix of this set -> swizzled smem, once
    const int chunks = NCHB * kblocks * 128 * 8;  // 16-byte chunks
    for (int id = tid; id < chunks; id += THREADS) {
      const int c = id & 7, r = (id >> 3) & 127, blk = id >> 10;  // blk = chb * kblocks + kb
      const int chb = blk / kblocks, kb = blk - chb * kblocks;
      const uint4 v = *reinterpret_cast<const uint4*>(W + (size_t)(chb * 128 + r) * g.ldw + kb * KB + c * 8);
      *reinterpret_cast<uint4*>(smem_gen + (size_t)blk * w_block_bytes + sw128(r, c)) = v;
    }
    fence_proxy_async();
  }
  if (GATHER) {
    float4* w1x = reinterpret_cast<float4*>(smem_gen + (w1x_base - smem_base));
    const float* src = g.W1x[wset];
    for (int k = tid; k < g.K; k += THREADS)
      w1x[k] = make_float4(src[(size_t)k * g.ldw1x], src[(size_t)k * g.ldw1x + 1], src[(size_t)k * g.ldw1x + 2], 0.f);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  if (warp >= EPI_WARPS + 1) {
    // =========================================================== producers
    const int pt = tid - (EPI_WARPS + 1) * 32;
    if (GATHER) {
      // X[r, k] = relu(P[rows[r], k] - Q[(row0+r)/32, k]).  The 256 producer threads form two groups that own
      // alternate stages.  A group gathers the raw bf16 rows of its NEXT stage with cp.async straight into the
      // swizzled operand slot (plus the stage's Q tile), and only then transforms its CURRENT stage in place
      // (each thread rewrites the 16-byte chunks it copied itself), so a whole stage of gathers per group is
      // always in flight while the other one is being converted -- the L2 round trip is off the critical path.
      constexpr int GCH = ROWS * 8 / 128;                  // 16-byte chunks per thread per stage
      constexpr int QCH = (ROWS / 32) * 8;                 // 16-byte chunks of the stage's Q tile ([groups][64] bf16)
      const int grp = pt >> 7, gt = pt & 127, gc = gt & 7, r0 = gt >> 3;
      int my_tiles = 0;
      for (int t = tile_begin + rank_in_set; t < tile_begin + tiles_per_set; t += step) ++my_tiles;
      const int jobs = my_tiles * kblocks;
      // the gathered row ids of a job are fetched one job ahead (into registers), so that the L2 round trip of the
      // index load is not in front of every stage's cp.async burst
      int src[GCH];
      auto fetch_ids = [&](int j) {
        const int ti = j / kblocks;
        const int row0 = (tile_begin + rank_in_set + ti * step) * ROWS;
#pragma unroll
        for (int i = 0; i < GCH; ++i) src[i] = g.rows[row0 + r0 + i * 16];
      };
      if (grp < jobs) fetch_ids(grp);
      auto issue = [&](int j) {
        const int ti = j / kblocks, kb = j - ti * kblocks;
        const int row0 = (tile_begin + rank_in_set + ti * step) * ROWS;      // ch_tiles == 1 in gather mode
        const uint32_t s = (uint32_t)j % NST, ph = ((uint32_t)j / NST) & 1;
        mbar_wait(empty_bar + 8 * s, ph ^ 1);
        const uint32_t st_addr = stages_base + s * STAGE_BYTES;
#pragma unroll
        for (int i = 0; i < GCH; ++i)
          cp_async16(st_addr + sw128(r0 + i * 16, gc), g.X + (size_t)src[i] * g.ldx + kb * KB + gc * 8);
        if (j + 2 < jobs) fetch_ids(j + 2);
        if (gt < (ROWS / 32) * 3) {   // the stage's group centres (fp32 xyz), 4-byte copies into a padded [g][4] tile
          const int gi = gt / 3, d = gt - gi * 3;
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(cstage_base + s * ((ROWS / 32) * 16) + gi * 16 + d * 4),
                       "l"(g.centers + (size_t)((row0 >> 5) + gi) * 3 + d)
                       : "memory");
        }
        cp_async_commit();
      };
      int j = grp;
      if (j < jobs) issue(j);
      long long* pprof = (pt == 0) ? g.prof : nullptr;   // group 0, thread 0
      for (; j < jobs; j += 2) {
        if (j < 48) tl_stamp(pprof, 1024 + (j >> 1) * 4);
        if (j + 2 < jobs) {
          issue(j + 2);
          cp_async_wait<1>();
        } else {
          cp_async_wait<0>();
        }
        // the centres were copied by other threads of the group
        asm volatile("bar.sync %0, 128;" ::"r"(2 + grp) : "memory");
        if (j < 48) tl_stamp(pprof, 1024 + (j >> 1) * 4 + 1);
        const uint32_t s = (uint32_t)j % NST;
        {  // Q[g][k] = W1[k,0:3] . centre_g for the 64 channels of this k-block: (ROWS/32)*64 values, 128 threads
          const int kb = j % kblocks;
          const float4* w1x = reinterpret_cast<const float4*>(smem_gen + (w1x_base - smem_base)) + kb * KB;
          const float4* cs = reinterpret_cast<const float4*>(smem_gen + (cstage_base + s * ((ROWS / 32) * 16) - smem_base));
          __nv_bfloat162* qt = reinterpret_cast<__nv_bfloat162*>(smem_gen + (qstage_base + s * (QCH * 16) - smem_base));
#pragma unroll
          for (int e = gt; e < (ROWS / 32) * 32; e += 128) {   // one bf16 pair per iteration
            const int gi = e >> 5, k2 = (e & 31) * 2;
            const float4 c = cs[gi], wa = w1x[k2], wb = w1x[k2 + 1];
            qt[e] = __floats2bfloat162_rn(fmaf(wa.x, c.x, fmaf(wa.y, c.y, wa.z * c.z)),
                                          fmaf(wb.x, c.x, fmaf(wb.y, c.y, wb.z * c.z)));
          }
        }
        asm volatile("bar.sync %0, 128;" ::"r"(2 + grp) : "memory");
        if (j < 48) tl_stamp(pprof, 1024 + (j >> 1) * 4 + 2);
        uint8_t* st_gen = smem_gen + (stages_base + s * STAGE_BYTES - smem_base);
        // packed bf16x2 arithmetic: relu(p - q) on two channels per instruction (HFMA2.BF16 rounds once)
        const uint4* qs = reinterpret_cast<const uint4*>(smem_gen + (qstage_base + s * (QCH * 16) - smem_base));
        const __nv_bfloat162 zero2 = __floats2bfloat162_rn(0.f, 0.f);
#pragma unroll
        for (int i = 0; i < GCH; i += 2) {   // chunks i and i+1 are rows r0+16i, r0+16(i+1): the same group of 32
          const int r = r0 + i * 16;
          const uint4 qv = qs[(r >> 5) * 8 + gc];
          const __nv_bfloat162* q2 = reinterpret_cast<const __nv_bfloat162*>(&qv);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            uint4* slot = reinterpret_cast<uint4*>(st_gen + sw128(r + h * 16, gc));
            uint4 pv = *slot;
            __nv_bfloat162* p2 = reinterpret_cast<__nv_bfloat162*>(&pv);
#pragma unroll
            for (int e = 0; e < 4; ++e) p2[e] = __hmax2(__hsub2(p2[e], q2[e]), zero2);
            *slot = pv;
          }
        }
        fence_proxy_async();
        mbar_arrive(full_bar + 8 * s);
        if (j < 48) tl_stamp(pprof, 1024 + (j >> 1) * 4 + 3);
        // a second group barrier keeps a fast thread from overwriting the Q tile of a slot that slower
        // threads of the group are still reading (slot s is reused by this group's job j + 2*NST at the earliest,
        // which is issued two iterations later -- so one barrier per iteration is enough)
      }
    } else {
    uint32_t issued = 0, arrived = 0;
    for (int t = tile_begin + rank_in_set; t < tile_begin + tiles_per_set; t += step) {
      const int cht = t % ch_tiles, rt = t / ch_tiles;
      const int row0 = rt * ROWS;
      for (int kb = 0; kb < kblocks; ++kb) {
        const uint32_t s = issued % NST;
        {
          const uint32_t ph = (issued / NST) & 1;
          mbar_wait(empty_bar + 8 * s, ph ^ 1);
          const uint32_t st_addr = stages_base + s * STAGE_BYTES;
          if (!RESIDENT) {
            for (int id = pt; id < NCHB * 128 * 8; id += PROD_THREADS) {
              const int c = id & 7, r = (id >> 3) & 127, chb = id >> 10;
              cp_async16(st_addr + chb * w_block_bytes + sw128(r, c),
                         W + (size_t)((cht * NCHB + chb) * 128 + r) * g.ldw + kb * KB + c * 8);
            }
          }
          for (int id = pt; id < ROWS * 8; id += PROD_THREADS) {
            const int c = id & 7, r = id >> 3;
            cp_async16(st_addr + STAGE_W_BYTES + sw128(r, c), g.X + (size_t)(row0 + r) * g.ldx + kb * KB + c * 8);
          }
          cp_async_commit();
          ++issued;
          if (issued - arrived > 2) {  // keep two stages of loads in flight
            cp_async_wait<2>();
            fence_proxy_async();
            mbar_arrive(full_bar + 8 * (arrived % NST));
            ++arrived;
          }
        }
      }
    }
    cp_async_wait<0>();
    fence_proxy_async();
    while (arrived < issued) {
      mbar_arrive(full_bar + 8 * (arrived % NST));
      ++arrived;
    }
    }
  } else if (warp == EPI_WARPS) {
    // =========================================================== MMA issuer (one thread)
    if (lane == 0) {
      const uint32_t idesc = make_idesc(ROWS);
      uint32_t it = 0, tc_count = 0;
      for (int t = tile_begin + rank_in_set; t < tile_begin + tiles_per_set; t += step, ++tc_count) {
        const uint32_t buf = tc_count & 1, aph = (tc_count >> 1) & 1;
        mbar_wait(acce_bar + 8 * buf, aph ^ 1);   // epilogue has drained this accumulator
        tc_fence_after();
        for (int kb = 0; kb < kblocks; ++kb, ++it) {
          const uint32_t s = it % NST, ph = (it / NST) & 1;
          mbar_wait(full_bar + 8 * s, ph);
          tc_fence_after();
          if (GATHER && it < 48) tl_stamp(g.prof, 1280 + it);
          const uint32_t st_addr = stages_base + s * STAGE_BYTES;
#pragma unroll
          for (int chb = 0; chb < NCHB; ++chb) {
            const uint32_t a_addr = RESIDENT ? smem_base + (uint32_t)(chb * kblocks + kb) * w_block_bytes
                                             : st_addr + chb * w_block_bytes;
            const uint64_t adesc = make_desc(a_addr), bdesc = make_desc(st_addr + STAGE_W_BYTES);
            const uint32_t d_tmem = tmem_base + (buf * NCHB + chb) * ROWS;
#pragma unroll
            for (int k4 = 0; k4 < KB / 16; ++k4)   // +32 bytes per UMMA_K=16 step inside the swizzle row
              umma_bf16(d_tmem, adesc + 2 * k4, bdesc + 2 * k4, idesc, (kb | k4) != 0);
          }
          umma_commit(empty_bar + 8 * s);          // stage reusable once these MMAs have read it
        }
        umma_commit(accf_bar + 8 * buf);           // accumulator complete
      }
    }
  } else {
    // =========================================================== epilogue (warps 0-3, TMEM lane = channel)
    uint32_t tc_count = 0;
    const int quarter = warp & 3, half = warp >> 2;            // half is 0 when there are only 4 epilogue warps
    constexpr int HALVES = EPI_WARPS / 4;
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    for (int t = tile_begin + rank_in_set; t < tile_begin + tiles_per_set; t += step, ++tc_count) {
      const int cht = t % ch_tiles, rt = t / ch_tiles;
      const int row0 = rt * ROWS;
      const uint32_t buf = tc_count & 1, aph = (tc_count >> 1) & 1;
      if (g.xyz) {   // coordinates of the tile's rows -> smem (coalesced), read back as broadcasts
        asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");   // previous tile's readers are done
        for (int i = tid; i < ROWS * 3; i += EPI_WARPS * 32) sxyz[i] = g.xyz[(size_t)row0 * 3 + i];
        asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
      }
      mbar_wait(accf_bar + 8 * buf, aph);
      tc_fence_after();
      if (GATHER && tid == 0 && tc_count < 24) tl_stamp(g.prof, 1408 + tc_count * 2);
#pragma unroll 1
      for (int chb = 0; chb < NCHB; ++chb) {
        const int ch = (cht * NCHB + chb) * 128 + quarter * 32 + lane;
        const bool ch_ok = g.n_valid <= 0 || ch < g.n_valid;
        const float bv = (bias && ch_ok) ? bias[ch] : 0.f;
        float tmax = -INFINITY;
        float w1x = 0.f, w1y = 0.f, w1z = 0.f;
        if (g.xyz) {
          const float* wp = g.W1x[wset] + (size_t)ch * g.ldw1x;
          w1x = wp[0]; w1y = wp[1]; w1z = wp[2];
        }
        const uint32_t t_addr = tmem_base + lane_base + (buf * NCHB + chb) * ROWS;
        float cmax = -INFINITY;
        // store epilogue: the two warps of a lane quarter take alternate chunks; max epilogues run on half 0 only
        const int c_begin = g.epi == 0 ? half : (half == 0 ? 0 : ROWS / 32);
        const int c_step = g.epi == 0 ? HALVES : 1;
        if (g.epi != 0 && half == 0) {
          // max epilogues: 64 accumulator columns (two neighbourhoods of 32 rows) per tcgen05.ld, each reduced by a
          // tree (depth 5, not a 31-long dependent chain): this loop paces the whole gather pipeline
#pragma unroll 1
          for (int c64 = 0; c64 < ROWS / 64; ++c64) {
            float v[64];
            tmem_ld64(t_addr + c64 * 64, v);
#pragma unroll
            for (int w = 32; w >= 2; w >>= 1) {
#pragma unroll
              for (int i = 0; i < w / 2; ++i) {
                v[i] = fmaxf(v[i], v[i + w / 2]);
                v[32 + i] = fmaxf(v[32 + i], v[32 + i + w / 2]);
              }
            }
            if (g.epi == 1) {  // one output row per group of 32
#pragma unroll
              for (int h = 0; h < 2; ++h) {
                float x = v[32 * h] + bv;
                if (g.relu) x = fmaxf(x, 0.f);
                const size_t grow = (size_t)(row0 >> 5) + c64 * 2 + h;
                if (g.Yf) g.Yf[grow * g.ldyf + ch] = x;
                if (g.Yb) g.Yb[grow * g.ldyb + ch] = __float2bfloat16_rn(x);
              }
            } else {
              cmax = fmaxf(cmax, fmaxf(v[0], v[32]));
            }
          }
        }
        // the store epilogue is compiled out of the gather kernels (launch_tc_gemm_gather allows the group max only):
        // it would cost them registers, and at the 128-register cap a spill
#pragma unroll 1
        for (int c32 = c_begin; c32 < ROWS / 32 && !GATHER && g.epi == 0; c32 += c_step) {
          float v[32];
          tmem_ld32(t_addr + c32 * 32, v);
          if (g.epi == 0) {
            // all residual loads of the chunk are issued before the first dependent use / store, so
            // their latency overlaps (one exposed L2 round trip per 32 rows instead of per row)
            const size_t rbase = (size_t)row0 + c32 * 32;
            if (!ch_ok) continue;                  // padded channel: nothing to store
            const float rbv = g.rowbias ? g.rowbias[(rbase / g.rb_rows) * g.rb_ld + ch] : 0.f;
            float res[32];
            if (g.Rf) {
              const float* rp = g.Rf + rbase * g.ldrf + ch;
#pragma unroll
              for (int i = 0; i < 32; ++i, rp += g.ldrf) res[i] = *rp;
            } else if (g.Rb) {
              const __nv_bfloat16* rp = g.Rb + rbase * g.ldrb + ch;
#pragma unroll
              for (int i = 0; i < 32; ++i, rp += g.ldrb) res[i] = __bfloat162float(*rp);
            }
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              float x = v[i] + bv + rbv;
              if (g.xyz) {
                const float* p = sxyz + (c32 * 32 + i) * 3;     // tile's coordinates staged in smem
                x = fmaf(w1x, p[0], fmaf(w1y, p[1], fmaf(w1z, p[2], x)));
              }
              if (g.relu) x = fmaxf(x, 0.f);
              if (g.Rf || g.Rb) x += res[i];
              v[i] = x;
              tmax = fmaxf(tmax, x);
            }
            if (g.Yf) {
              float* yp = g.Yf + rbase * g.ldyf + ch;
#pragma unroll
              for (int i = 0; i < 32; ++i, yp += g.ldyf) *yp = v[i];
            }
            if (g.Yb) {
              __nv_bfloat16* yp = g.Yb + rbase * g.ldyb + ch;
#pragma unroll
              for (int i = 0; i < 32; ++i, yp += g.ldyb) *yp = __float2bfloat16_rn(v[i]);
            }
          }
        }
        if (g.epi == 0 && g.Ymax && ch_ok) g.Ymax[((size_t)rt * 2 + half) * g.ldmax + ch] = tmax;   // 2 partials per tile
        if (g.epi == 2 && half == 0) {  // max over all ROWS rows of the tile (one cloud)
          float x = cmax + bv;
          if (g.relu) x = fmaxf(x, 0.f);
          if (g.Yf) g.Yf[(size_t)rt * g.ldyf + ch] = x;
        }
      }
      tc_fence_before();
      mbar_arrive(acce_bar + 8 * buf);
      if (GATHER && tid == 0 && tc_count < 24) tl_stamp(g.prof, 1408 + tc_count * 2 + 1);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == EPI_WARPS) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

template <int ROWS, int NCHB, bool RESIDENT, bool GATHER, int NST>
static int tc_launch(const TcGemm& g, cudaStream_t st) {
  const int kblocks = g.K / KB;
  const size_t resident = RESIDENT ? (size_t)NCHB * kblocks * 128 * 128 : 0;
  const size_t stage = (RESIDENT ? 0 : (size_t)NCHB * 128 * 128) + (size_t)ROWS * 128;
  const size_t smem = 1024 + resident + NST * stage + 8 * (2 * NST + 4) + 32 +
                      (GATHER ? (size_t)NST * (ROWS / 32) * (128 + 16) + (size_t)g.K * 16 : 0);
  PZ_REQUIRE(smem <= 227 * 1024, PZ_ERR_UNSUPPORTED, "tc_gemm: needs %zu B of shared memory (K=%d too large for a resident weight)", smem, g.K);
  auto kern = tc_gemm_kernel<ROWS, NCHB, RESIDENT, GATHER, NST>;
  PZ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int nsets = (g.rows_per_wset > 0 && g.M > g.rows_per_wset) ? 2 : 1;
  const int tiles = (g.M / ROWS) * (g.Nout / (128 * NCHB));
  int grid = tiles < kNumSMs ? tiles : kNumSMs;
  if (nsets == 2 && (grid & 1)) --grid;   // equal CTA count per weight set
  if (grid < nsets) grid = nsets;
  kern<<<grid, THREADS, smem, st>>>(g);
  PZ_LAUNCH_CHECK();
  return 0;
}

// gathered B operand, resident weights: stage 1 (Nout 128, 256-row tiles) and stage 2 (Nout 256, 128-row tiles)
static int launch_tc_gemm_gather(const TcGemm& g, cudaStream_t st, int nsets) {
  PZ_REQUIRE(g.centers && g.W1x[0] && g.epi == 1, PZ_ERR_ARG, "tc_gemm: gathered operand needs centres, W1x and the group-max epilogue");
  if (g.Nout == 128 && g.K <= 256) {
    PZ_REQUIRE(g.M % (256 * nsets) == 0, PZ_ERR_UNSUPPORTED, "tc_gemm: M=%d must be a multiple of %d", g.M, 256 * nsets);
    return tc_launch<256, 1, true, true, 4>(g, st);
  }
  if (g.Nout == 256 && g.K <= 256) {
    PZ_REQUIRE(g.M % (128 * nsets) == 0, PZ_ERR_UNSUPPORTED, "tc_gemm: M=%d must be a multiple of %d", g.M, 128 * nsets);
    return tc_launch<128, 2, true, true, 5>(g, st);
  }
  return fail(PZ_ERR_UNSUPPORTED, "tc_gemm: gathered GEMM supports (Nout,K) in {(128,<=256),(256,<=256)} (got %d,%d)", g.Nout, g.K);
}

int launch_tc_gemm(const TcGemm& g, cudaStream_t st) {
  PZ_REQUIRE(g.W[0] && g.X && (g.Yf || g.Yb), PZ_ERR_ARG, "tc_gemm: null operand");
  PZ_REQUIRE(g.M > 0 && g.Nout > 0 && g.K > 0, PZ_ERR_ARG, "tc_gemm: bad shape");
  PZ_REQUIRE(g.K % 64 == 0 && g.Nout % 128 == 0 && g.ldx % 8 == 0 && g.ldw % 8 == 0, PZ_ERR_UNSUPPORTED,
             "tc_gemm: needs K %% 64 == 0, Nout %% 128 == 0 and 16-byte aligned rows (K=%d Nout=%d)", g.K, g.Nout);
  PZ_REQUIRE(((uintptr_t)g.X & 15) == 0 && ((uintptr_t)g.W[0] & 15) == 0 && (!g.W[1] || ((uintptr_t)g.W[1] & 15) == 0),
             PZ_ERR_ARG, "tc_gemm: operands must be 16-byte aligned");
  const int nsets = (g.rows_per_wset > 0 && g.M > g.rows_per_wset) ? 2 : 1;
  if (nsets == 2) PZ_REQUIRE(g.W[1] && g.M == 2 * g.rows_per_wset, PZ_ERR_ARG, "tc_gemm: two weight sets need M == 2*rows_per_wset");
  if (g.rows) {
    TcGemm gp = g;   // diagnostics: only the stage-1 variant stamps, so one forward leaves one timeline
    gp.prof = (g.Nout == 128) ? kernel_timeline_buffer(1456) : nullptr;   // slots 1024..1455
    return launch_tc_gemm_gather(gp, st, nsets);
  }
  PZ_REQUIRE(g.M % (256 * nsets) == 0, PZ_ERR_UNSUPPORTED, "tc_gemm: M=%d must be a multiple of %d", g.M, 256 * nsets);
  return tc_launch<256, 1, false, false, 4>(g, st);
}

// fp32 -> bf16 with row strides (weights packs, activations entering the tensor-core path)
__global__ void __launch_bounds__(256) cvt_bf16_kernel(const float* __restrict__ in, int ldi, int rows, int cols,
                                                       __nv_bfloat16* __restrict__ out, int ldo) {
  const size_t total = (size_t)rows * cols;
  for (size_t e = (size_t)blockIdx.x * 256 + threadIdx.x; e < total; e += (size_t)gridDim.x * 256) {
    const size_t r = e / cols;
    const int c = (int)(e - r * cols);
    out[r * ldo + c] = __float2bfloat16_rn(in[r * ldi + c]);
  }
}

int launch_cvt_bf16(const float* in, int ldi, int rows, int cols, __nv_bfloat16* out, int ldo, cudaStream_t st) {
  const size_t total = (size_t)rows * cols;
  if (total == 0) return 0;
  const int blocks = (int)((total + 255) / 256 < (size_t)kNumSMs * 8 ? (total + 255) / 256 : (size_t)kNumSMs * 8);
  cvt_bf16_kernel<<<blocks, 256, 0, st>>>(in, ldi, rows, cols, out, ldo);
  PZ_LAUNCH_CHECK();
  return 0;
}

}  // namespace pz

using namespace pz;

extern "C" int pz_linear_bf16(const void* x_bf16, int ldx, const void* w_bf16, const float* bias, int M, int N, int K,
                              int relu, const float* residual_or_null, int ldr, float* y, int ldy, pz_stream_t stream) {
  PZ_REQUIRE(x_bf16 && w_bf16 && y, PZ_ERR_ARG, "pz_linear_bf16: null pointer");
  PZ_REQUIRE(M >= 0 && N >= 1 && K >= 1 && ldx >= K && ldy >= N, PZ_ERR_ARG, "pz_linear_bf16: bad sizes");
  if (M == 0) return 0;
  TcGemm g;
  g.X = static_cast<const __nv_bfloat16*>(x_bf16); g.ldx = ldx;
  g.W[0] = static_cast<const __nv_bfloat16*>(w_bf16); g.ldw = K; g.bias[0] = bias;
  g.M = M; g.Nout = N; g.K = K; g.relu = relu; g.Yf = y; g.ldyf = ldy; g.Rf = residual_or_null; g.ldrf = ldr;
  return launch_tc_rowgemm(g, as_stream(stream));
}
