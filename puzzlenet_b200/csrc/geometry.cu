// Point-cloud geometry kernels for sm_100a: farthest-point sampling, kNN selection,
// square_distance, ball query, row gather and the materialising grouping of
// sample_and_group.  Reference semantics: pointnet_util.py:22-136.
//
// Arithmetic contract (bit-exact indices): every squared distance is
//   ((dx*dx) + (dy*dy)) + (dz*dz)   in fp32, each op rounded, no FMA contraction
// (the ATen CPU evaluation of pointnet_util.py:36 / :70), hence the explicit
// __fmul_rn / __fadd_rn below.
#include <stdlib.h>

#include "pz_common.cuh"

namespace pz {

__device__ __forceinline__ float sqdist3(float ax, float ay, float az, float bx, float by, float bz) {
  float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
  return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

// ======================================================================================
// Farthest point sampling: one CTA per cloud, cloud + running min-distance in registers
// (PPT points per thread, strided so that a thread's points are in increasing index
// order), coordinates mirrored in shared memory (SoA) for the centroid broadcast.
// One __syncthreads per iteration: warp argmax with two redux.sync, per-warp winners in a
// parity-double-buffered smem slot, every warp re-reduces the <=32 winners redundantly.
// Key = (dist_bits << 32) | ~index: max key == largest distance, lowest index on ties
// (torch.max on CPU returns the first maximum, pointnet_util.py:72).
// ======================================================================================
template <int PPT, int T>
__global__ void __launch_bounds__(T) fps_kernel(const float* __restrict__ xyz, int N, int S,
                                                const int64_t* __restrict__ start,
                                                int64_t* __restrict__ out64,
                                                int* __restrict__ out_rows32,
                                                float* __restrict__ new_xyz) {
  extern __shared__ float fps_smem[];
  float* xs = fps_smem;
  float* ys = xs + N;
  float* zs = ys + N;
  int* sel = reinterpret_cast<int*>(zs + N);   // [S] picked indices; written out coalesced after the loop
  __shared__ unsigned int whi[2][32];
  __shared__ unsigned int wlo[2][32];

  const int c = blockIdx.x;
  const int t = threadIdx.x;
  const int lane = t & 31, warp = t >> 5;
  pdl_enter();
  const float* p = xyz + (size_t)c * N * 3;
  for (int i = t; i < N * 3; i += T) {
    float v = p[i];
    int pt = i / 3, d = i - pt * 3;
    fps_smem[d * N + pt] = v;
  }
  if (t < 64) (&whi[0][0])[t] = 0u, (&wlo[0][0])[t] = 0u;   // slots of absent warps stay 0 = "no candidate"
  __syncthreads();

  // Padding slots (index >= N) sit at the origin with min-distance 0: fminf(0, d) stays 0, so they need no
  // bounds test in the loop and can never beat a real point (ties resolve to the lowest index).
  float px[PPT], py[PPT], pz_[PPT], md[PPT];
#pragma unroll
  for (int j = 0; j < PPT; ++j) {
    int i = t + j * T;
    bool ok = i < N;
    px[j] = ok ? xs[i] : 0.f;
    py[j] = ok ? ys[i] : 0.f;
    pz_[j] = ok ? zs[i] : 0.f;
    md[j] = ok ? 1e10f : 0.f;
  }

  int far = (int)start[c];
  far = min(max(far, 0), N - 1);
  for (int s = 0; s < S; ++s) {
    if (t == 0) sel[s] = far;
    if (s + 1 == S) break;
    const float cx = xs[far], cy = ys[far], cz = zs[far];
    float best = -1.f;
    int bestj = 0;
#pragma unroll
    for (int j = 0; j < PPT; ++j) {
      md[j] = fminf(md[j], sqdist3(px[j], py[j], pz_[j], cx, cy, cz));
      const bool gt = md[j] > best;   // strict: the earlier (lower) index wins inside a thread
      best = gt ? md[j] : best;
      bestj = gt ? j : bestj;
    }
    const unsigned int hi = __float_as_uint(best);  // distances are >= 0: the bit pattern is order preserving
    const unsigned int lo = ~(unsigned int)(t + bestj * T);
    const unsigned int mhi = __reduce_max_sync(0xffffffffu, hi);
    const unsigned int mlo = __reduce_max_sync(0xffffffffu, hi == mhi ? lo : 0u);
    const int par = s & 1;
    if (lane == 0) {
      whi[par][warp] = mhi;
      wlo[par][warp] = mlo;
    }
    __syncthreads();
    const unsigned int h2 = whi[par][lane];
    const unsigned int l2 = wlo[par][lane];
    const unsigned int ghi = __reduce_max_sync(0xffffffffu, h2);
    const unsigned int glo = __reduce_max_sync(0xffffffffu, h2 == ghi ? l2 : 0u);
    far = (int)(~glo);
  }
  __syncthreads();
  for (int s = t; s < S; s += T) {
    const int f = sel[s];
    const size_t o = (size_t)c * S + s;
    if (out64) out64[o] = f;
    if (out_rows32) out_rows32[o] = c * N + f;
    if (new_xyz) {
      new_xyz[o * 3 + 0] = xs[f];
      new_xyz[o * 3 + 1] = ys[f];
      new_xyz[o * 3 + 2] = zs[f];
    }
  }
}

template <int PPT, int T>
static int fps_launch_t(const float* xyz, int B, int N, const int64_t* start, int S, int64_t* out64,
                        int* out_rows32, float* new_xyz, cudaStream_t st) {
  size_t smem = (size_t)N * 3 * sizeof(float) + (size_t)S * sizeof(int);
  PZ_REQUIRE(smem <= 227 * 1024, PZ_ERR_UNSUPPORTED, "pz_fps: N=%d, S=%d need %zu B of shared memory", N, S, smem);
  if (smem > 48 * 1024)
    PZ_CUDA(cudaFuncSetAttribute(fps_kernel<PPT, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  PZ_CUDA(launch_pdl(fps_kernel<PPT, T>, dim3(B), dim3(T), smem, st, xyz, N, S, start, out64, out_rows32, new_xyz));
  PZ_LAUNCH_CHECK();
  return 0;
}

// ---- large clouds (dataset shape, 11000 -> 1024): a thread-block cluster of CS = 2 or 4 CTAs per cloud.  Each CTA keeps
// the running minimum distances of 1/CS of the points in registers (the per-iteration update -- 32 warps x PPT points x
// ~12 instructions, issue bound -- shrinks by CS) and the whole cloud's coordinates in its own shared memory (the centroid
// lookup stays local).  Per iteration the CTAs exchange ONE 64-bit key each (distance bits, ~index): a thread per peer
// sends its CTA's winner into its slot at that peer with st.async, which also completes the transaction count of the
// peer's mbarrier; every thread then waits on its own CTA's mbarrier and takes the largest key.  No cluster-wide barrier inside the loop
// (cluster.sync costs ~380 cycles and flushes L1; the mbarrier round trip is one DSMEM store).
__device__ __forceinline__ uint32_t fps_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
template <int PPT, int CS>
__global__ void __launch_bounds__(1024) fps_cluster_kernel(const float* __restrict__ xyz, int N, int S,
                                                           const int64_t* __restrict__ start, int64_t* __restrict__ out64,
                                                           int* __restrict__ out_rows32, float* __restrict__ new_xyz) {
  constexpr int T = 1024;
  extern __shared__ float fps_smem[];
  float* xs = fps_smem;
  float* ys = xs + N;
  float* zs = ys + N;
  int* sel = reinterpret_cast<int*>(zs + N);
  __shared__ unsigned int whi[2][32];
  __shared__ unsigned int wlo[2][32];
  __shared__ __align__(8) unsigned long long peer_key[2][CS]; // slot [parity][sender rank], written by the PEER CTAs (st.async)
  __shared__ __align__(8) unsigned long long xbar[2];         // mbarriers completed by the peers' st.async

  const int c = blockIdx.x / CS;
  unsigned int rank;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
  const int t = threadIdx.x;
  const int lane = t & 31, warp = t >> 5;
  const float* p = xyz + (size_t)c * N * 3;
  for (int i = t; i < N * 3; i += T) {
    float v = p[i];
    int pt = i / 3, d = i - pt * 3;
    fps_smem[d * N + pt] = v;
  }
  if (t < 64) (&whi[0][0])[t] = 0u, (&wlo[0][0])[t] = 0u;
  if (t == 0) {
    for (int b = 0; b < 2; ++b)
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(fps_smem_u32(&xbar[b])) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  // both CTAs have initialised their barriers before anyone sends
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
  // lanes 1 .. CS-1 of warp 0 each own one peer: the peer's copy of my slot in ITS peer_key and of its barriers
  uint32_t remote_key[2] = {0, 0}, remote_bar[2] = {0, 0};
  if (t >= 1 && t < CS) {
    const unsigned int peer = (rank + t) % CS;
    for (int b = 0; b < 2; ++b) {
      asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote_key[b]) : "r"(fps_smem_u32(&peer_key[b][rank])), "r"(peer));
      asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote_bar[b]) : "r"(fps_smem_u32(&xbar[b])), "r"(peer));
    }
  }

  const int part = (N + CS - 1) / CS;                          // contiguous index ranges: CTA r owns [r*part, min(N, (r+1)*part))
  const int base = (int)rank * part, cnt = max(0, min(N, base + part) - base);
  float px[PPT], py[PPT], pz_[PPT], md[PPT];
#pragma unroll
  for (int j = 0; j < PPT; ++j) {
    const int li = t + j * T;
    const bool ok = li < cnt;
    const int i = base + li;
    px[j] = ok ? xs[i] : 0.f;
    py[j] = ok ? ys[i] : 0.f;
    pz_[j] = ok ? zs[i] : 0.f;
    md[j] = ok ? 1e10f : 0.f;
  }

  int far = (int)start[c];
  far = min(max(far, 0), N - 1);
  for (int s = 0; s < S; ++s) {
    if (t == 0) sel[s] = far;
    if (s + 1 == S) break;
    const float cx = xs[far], cy = ys[far], cz = zs[far];
    float best = -1.f;
    int bestj = 0;
#pragma unroll
    for (int j = 0; j < PPT; ++j) {
      md[j] = fminf(md[j], sqdist3(px[j], py[j], pz_[j], cx, cy, cz));
      const bool gt = md[j] > best;
      best = gt ? md[j] : best;
      bestj = gt ? j : bestj;
    }
    const unsigned int hi = __float_as_uint(best);
    const unsigned int lo = ~(unsigned int)(base + t + bestj * T);
    const unsigned int mhi = __reduce_max_sync(0xffffffffu, hi);
    const unsigned int mlo = __reduce_max_sync(0xffffffffu, hi == mhi ? lo : 0u);
    const int par = s & 1;
    if (lane == 0) {
      whi[par][warp] = mhi;
      wlo[par][warp] = mlo;
    }
    __syncthreads();
    const unsigned int h2 = whi[par][lane];
    const unsigned int l2 = wlo[par][lane];
    const unsigned int ghi = __reduce_max_sync(0xffffffffu, h2);
    const unsigned int glo = __reduce_max_sync(0xffffffffu, h2 == ghi ? l2 : 0u);
    const unsigned long long mine = ((unsigned long long)ghi << 32) | glo;
    if (t == 0)      // arm my barrier for the peers' 8 bytes each
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(fps_smem_u32(&xbar[par])), "r"(8 * (CS - 1)) : "memory");
    else if (t < CS) // send my key into my slot at one peer (completes ITS barrier)
      asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];"
                   ::"r"(remote_key[par]), "l"(mine), "r"(remote_bar[par]) : "memory");
    {  // wait for the peer's key of this iteration (phase of barrier `par` = its use count parity)
      const uint32_t bar = fps_smem_u32(&xbar[par]), phase = (uint32_t)(s >> 1) & 1u;
      uint32_t ok = 0;
      for (uint32_t spin = 0; !ok; ++spin) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(phase) : "memory");
        if (!ok && spin > (1u << 24)) __trap();   // a protocol bug must be a launch failure, never a hang
      }
    }
    unsigned long long win = mine;
#pragma unroll
    for (int r = 0; r < CS; ++r) {
      const unsigned long long theirs = *reinterpret_cast<volatile unsigned long long*>(&peer_key[par][r]);
      if (r != (int)rank && theirs > win) win = theirs;
    }
    far = (int)(~(unsigned int)(win & 0xffffffffull));
  }
  __syncthreads();
  if (rank == 0) {
    for (int s = t; s < S; s += T) {
      const int f = sel[s];
      const size_t o = (size_t)c * S + s;
      if (out64) out64[o] = f;
      if (out_rows32) out_rows32[o] = c * N + f;
      if (new_xyz) {
        new_xyz[o * 3 + 0] = xs[f];
        new_xyz[o * 3 + 1] = ys[f];
        new_xyz[o * 3 + 2] = zs[f];
      }
    }
  }
  // neither CTA may exit while the other can still write into its shared memory
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

template <int PPT, int CS>
static int fps_launch_cluster(const float* xyz, int B, int N, const int64_t* start, int S, int64_t* out64,
                              int* out_rows32, float* new_xyz, cudaStream_t st) {
  size_t smem = (size_t)N * 3 * sizeof(float) + (size_t)S * sizeof(int);
  PZ_REQUIRE(smem <= 226 * 1024, PZ_ERR_UNSUPPORTED, "pz_fps: N=%d, S=%d need %zu B of shared memory", N, S, smem);
  PZ_CUDA(cudaFuncSetAttribute(fps_cluster_kernel<PPT, CS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(CS * B);
  cfg.blockDim = dim3(1024);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  PZ_CUDA(cudaLaunchKernelEx(&cfg, fps_cluster_kernel<PPT, CS>, xyz, N, S, start, out64, out_rows32, new_xyz));
  count_launch();
  return 0;
}

static int fps_grid_launch(const float* xyz, int B, int N, const int64_t* start, int S, int64_t* out64, int* out_rows32,
                           float* new_xyz, cudaStream_t st);   // large clouds: block-pruned updates (defined next to the grid kNN)

int launch_fps(const float* xyz, int B, int N, const int64_t* start, int S, int64_t* out64,
               int* out_rows32, float* new_xyz, cudaStream_t st) {
  if (N > 4096 && N <= 14336 && S <= 8192) return fps_grid_launch(xyz, B, N, start, S, out64, out_rows32, new_xyz, st);
  // large clouds, few enough of them that two CTAs per cloud still run in one wave: the 2-CTA cluster variant
  if (N > 4096 && 4 * B <= kNumSMs) {     // a handful of large clouds (assembly, dataset): 4 CTAs per cloud
    const int part = (N + 3) / 4;
    if (part <= 2 * 1024) return fps_launch_cluster<2, 4>(xyz, B, N, start, S, out64, out_rows32, new_xyz, st);
    if (part <= 3 * 1024) return fps_launch_cluster<3, 4>(xyz, B, N, start, S, out64, out_rows32, new_xyz, st);
    if (part <= 4 * 1024) return fps_launch_cluster<4, 4>(xyz, B, N, start, S, out64, out_rows32, new_xyz, st);
  }
  if (N > 4096 && 2 * B <= kNumSMs) {
    const int part = (N + 1) / 2;
    if (part <= 3 * 1024) return fps_launch_cluster<3, 2>(xyz, B, N, start, S, out64, out_rows32, new_xyz, st);
    if (part <= 4 * 1024) return fps_launch_cluster<4, 2>(xyz, B, N, start, S, out64, out_rows32, new_xyz, st);
    if (part <= 6 * 1024) return fps_launch_cluster<6, 2>(xyz, B, N, start, S, out64, out_rows32, new_xyz, st);
    if (part <= 8 * 1024) return fps_launch_cluster<8, 2>(xyz, B, N, start, S, out64, out_rows32, new_xyz, st);
  }
  if (N <= 256) return fps_launch_t<2, 128>(xyz, B, N, start, S, out64, out_rows32, new_xyz, st);
  if (N <= 512) return fps_launch_t<4, 128>(xyz, B, N, start, S, out64, out_rows32, new_xyz, st);
  if (N <= 1024) return fps_launch_t<4, 256>(xyz, B, N, start, S, out64, out_rows32, new_xyz, st);
  if (N <= 2048) return fps_launch_t<4, 512>(xyz, B, N, start, S, out64, out_rows32, new_xyz, st);
  if (N <= 4096) return fps_launch_t<4, 1024>(xyz, B, N, start, S, out64, out_rows32, new_xyz, st);
  if (N <= 8192) return fps_launch_t<8, 1024>(xyz, B, N, start, S, out64, out_rows32, new_xyz, st);
  if (N <= 16384) return fps_launch_t<16, 1024>(xyz, B, N, start, S, out64, out_rows32, new_xyz, st);
  return fail(PZ_ERR_UNSUPPORTED, "pz_fps: N=%d exceeds the supported maximum 16384", N);
}

// ======================================================================================
// kNN: one warp per query.  Keys are (distance bits, index) pairs, ordered by distance and
// then index.  The warp keeps its current best 32 keys sorted across lanes.  Per sub-chunk
// of 1024 candidates (32 per lane, distances kept in registers):
//   pass 1   distances + each lane's two smallest (m0 <= m1);
//   bound    the current 32nd distance if one is known, else a bisection on the bit pattern
//            for the smallest x (to 1/256 of [min m1, max m0]) with at least 32 of the 64
//            lane minima <= x: an upper bound of the true 32nd distance that typically admits
//            only ~36 candidates;
//   compact  every lane counts its candidates <= bound, one warp scan gives each lane its
//            slot range in the per-warp queue (no per-iteration ballots), the survivors are
//            written with predicated stores;
//   fold     first sub-chunk: one bitonic sort of 32 queue entries becomes the sorted list,
//            the few extra entries are inserted one by one (shift by shuffle); later
//            sub-chunks insert their few improvements the same way; more than 12 pending
//            entries go through the bitonic sort + merge network 32 at a time.
// More than 64 candidates under the bound (heavy distance ties) take the incremental path:
// ballot compaction with a merge whenever the queue fills.  The [B,S,N] distance matrix of
// pointnet_util.py:118 never exists.
// ======================================================================================
constexpr int KNN_WARPS = 8;      // warps per CTA
constexpr int KNN_QPW = 4;        // queries per warp (amortises staging the cloud in shared memory)
constexpr int KNN_CHUNK = 2048;   // points staged in smem per pass
constexpr int KNN_PSTRIDE = KNN_CHUNK + 4;   // x / y / z planes, offset by 4 banks so the AoS -> SoA staging stores spread

__device__ __forceinline__ void knn_merge_inl(unsigned& td, unsigned& ti, unsigned cd, unsigned ci, int lane, unsigned kmask);
// Out-of-line wrappers: the networks are ~120 / ~200 instructions and are reached from inside unrolled
// candidate loops; one shared copy keeps the kernel inside the instruction cache.
__device__ __noinline__ uint2 knn_merge_call(unsigned td, unsigned ti, unsigned cd, unsigned ci, int lane, unsigned kmask);
__device__ __noinline__ uint2 knn_sort_call(unsigned cd, unsigned ci, unsigned kmask);
__device__ __forceinline__ void knn_merge(unsigned& td, unsigned& ti, unsigned cd, unsigned ci, int lane, unsigned kmask) {
  const uint2 r = knn_merge_call(td, ti, cd, ci, lane, kmask);
  td = r.x;
  ti = r.y;
}

// (distance bits, index) pairs kept in two 32-bit registers; order = distance, then index
__device__ __forceinline__ bool key_less(unsigned ad, unsigned ai, unsigned bd, unsigned bi) {
  return ad < bd || (ad == bd && ai < bi);
}
// one compare-exchange stage of a bitonic network across the warp; keep_min: this lane keeps the smaller key
__device__ __forceinline__ void cx_stage(unsigned& d, unsigned& i, int j, bool keep_min) {
  const unsigned od = __shfl_xor_sync(0xffffffffu, d, j), oi = __shfl_xor_sync(0xffffffffu, i, j);
  const bool take = key_less(od, oi, d, i) == keep_min;
  d = take ? od : d;
  i = take ? oi : i;
}
// kmask bit s = keep_min of this lane in sort stage s (the 15 stages of a 32-wide bitonic sort, in order)
__device__ __forceinline__ unsigned bitonic_keep_mask(int lane) {
  unsigned m = 0;
  int s = 0;
  for (int k = 2; k <= 32; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1, ++s) {
      const bool asc = (lane & k) == 0 || k == 32;
      if (((lane & j) == 0) == asc) m |= 1u << s;
    }
  return m;
}
// 32 keys (one per lane, any order) -> ascending across lanes
__device__ __forceinline__ void knn_sort_inl(unsigned& cd, unsigned& ci, unsigned kmask) {
  int s = 0;
#pragma unroll
  for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1, ++s) cx_stage(cd, ci, j, (kmask >> s) & 1u);
  }
}
// fold 32 candidate keys (one per lane, any order) into the sorted top-32 (td, ti)
__device__ __forceinline__ void knn_merge_inl(unsigned& td, unsigned& ti, unsigned cd, unsigned ci, int lane, unsigned kmask) {
  knn_sort_inl(cd, ci, kmask);
  const unsigned rd = __shfl_sync(0xffffffffu, cd, 31 - lane), ri = __shfl_sync(0xffffffffu, ci, 31 - lane);
  const bool lt = key_less(rd, ri, td, ti);   // elementwise min of ascending top and descending candidates:
  td = lt ? rd : td;                          // a bitonic sequence holding the 32 smallest of the union
  ti = lt ? ri : ti;
#pragma unroll
  for (int j = 16, q = 10; j > 0; j >>= 1, ++q) cx_stage(td, ti, j, (kmask >> q) & 1u);   // = the k == 32 stages
}

__device__ __noinline__ uint2 knn_merge_call(unsigned td, unsigned ti, unsigned cd, unsigned ci, int lane, unsigned kmask) {
  knn_merge_inl(td, ti, cd, ci, lane, kmask);
  return make_uint2(td, ti);
}
__device__ __noinline__ uint2 knn_sort_call(unsigned cd, unsigned ci, unsigned kmask) {
  knn_sort_inl(cd, ci, kmask);
  return make_uint2(cd, ci);
}
// insert one key (the same in every lane) into the ascending list: lanes past its place shift up by one
__device__ __forceinline__ void knn_insert(unsigned& td, unsigned& ti, unsigned xd, unsigned xi, int lane) {
  const unsigned pd = __shfl_up_sync(0xffffffffu, td, 1), pi = __shfl_up_sync(0xffffffffu, ti, 1);
  const bool lt = key_less(xd, xi, td, ti);
  const bool ltp = lane > 0 && key_less(xd, xi, pd, pi);
  td = lt ? (ltp ? pd : xd) : td;
  ti = lt ? (ltp ? pi : xi) : ti;
}

__global__ void __launch_bounds__(KNN_WARPS * 32, 3) knn_kernel(const float* __restrict__ query,
                                                             const float* __restrict__ xyz, int S,
                                                             int N, int K,
                                                             int64_t* __restrict__ out64,
                                                             int* __restrict__ out_rows32,
                                                             float* __restrict__ out_d2) {
  // the cloud is staged as x / y / z planes: lane l reads points 4(32 t + l) .. +3 of a sub-chunk with three
  // 128-bit loads
  __shared__ __align__(16) float pts[3 * KNN_PSTRIDE];
  __shared__ uint2 qkey[KNN_WARPS][64];   // per-warp candidate queue: (distance bits, index)
  const int b = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int q0 = (blockIdx.x * KNN_WARPS + warp) * KNN_QPW;
  const float* p = xyz + (size_t)b * N * 3;
  const unsigned kmask = bitonic_keep_mask(lane);
  uint2* myq = qkey[warp];
  const unsigned lt_mask = (1u << lane) - 1u;
  // per-query selection state lives in registers while the query is being scanned and is parked in shared
  // memory between chunks (only clouds larger than KNN_CHUNK points have more than one chunk); the query loop
  // is deliberately not unrolled so that the networks are emitted once (instruction-cache footprint)
  __shared__ unsigned park_d[KNN_WARPS][KNN_QPW][32], park_i[KNN_WARPS][KNN_QPW][32];
  pdl_enter();

  for (int base = 0; base < N; base += KNN_CHUNK) {
    const int cnt = min(KNN_CHUNK, N - base);
    const bool first = base == 0, last = base + KNN_CHUNK >= N;
    __syncthreads();
    for (int i = threadIdx.x; i < cnt * 3; i += KNN_WARPS * 32) {
      const int pi = i / 3;
      pts[(i - 3 * pi) * KNN_PSTRIDE + pi] = p[(size_t)base * 3 + i];
    }
    // the tail of the last 1024-candidate sub-chunk is filled with far-away points (distance ~3e36, index >= N):
    // they order after every real point, so they can only surface past the N-th neighbour, which K <= N never reads
    for (int i = cnt + threadIdx.x; i < ((cnt + 1023) & ~1023); i += KNN_WARPS * 32)
      pts[i] = pts[KNN_PSTRIDE + i] = pts[2 * KNN_PSTRIDE + i] = 1e18f;
    __syncthreads();
#pragma unroll 1
    for (int w = 0; w < KNN_QPW; ++w) {
      const int q = q0 + w;
      if (q >= S) break;                  // warp-uniform
      const float* qp = query + ((size_t)b * S + q) * 3;
      const float qx = qp[0], qy = qp[1], qz = qp[2];
      unsigned td = first ? 0xffffffffu : park_d[warp][w][lane];   // lane l holds the l-th smallest key so far
      unsigned ti = first ? 0xffffffffu : park_i[warp][w][lane];
      unsigned tau = __shfl_sync(0xffffffffu, td, 31);              // distance bits of the current 32nd smallest
#pragma unroll 1
      for (int sub = 0; sub < cnt; sub += 1024) {
        unsigned db[32];   // db[4 t4 + j] = candidate sub + 4 (32 t4 + lane) + j
        unsigned m0 = 0xffffffffu, m1 = 0xffffffffu;
#pragma unroll
        for (int t4 = 0; t4 < 8; ++t4) {
          const int i0 = sub + (t4 * 32 + lane) * 4;
          const float4 X = *reinterpret_cast<const float4*>(pts + i0);
          const float4 Y = *reinterpret_cast<const float4*>(pts + KNN_PSTRIDE + i0);
          const float4 Z = *reinterpret_cast<const float4*>(pts + 2 * KNN_PSTRIDE + i0);
          const float xs[4] = {X.x, X.y, X.z, X.w}, ys[4] = {Y.x, Y.y, Y.z, Y.w}, zs[4] = {Z.x, Z.y, Z.z, Z.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const unsigned x = __float_as_uint(sqdist3(qx, qy, qz, xs[j], ys[j], zs[j]));
            db[t4 * 4 + j] = x;
            m1 = min(m1, max(m0, x));
            m0 = min(m0, x);
          }
        }
        unsigned thr = tau;
        if (thr == 0xffffffffu) {   // warp-uniform
          unsigned hi = __reduce_max_sync(0xffffffffu, m0);   // >= 32 candidates are <= the largest lane minimum
          unsigned lo = __reduce_min_sync(0xffffffffu, m1);
          if (lo < hi) {
#pragma unroll 1
            for (int it = 0; it < 8 && lo < hi; ++it) {
              const unsigned mid = lo + ((hi - lo) >> 1);
              const int c = __reduce_add_sync(0xffffffffu, (m0 <= mid ? 1 : 0) + (m1 <= mid ? 1 : 0));
              if (c >= 32) hi = mid; else lo = mid + 1;
            }
          }
          thr = hi;
        }
        thr = min(thr, 0xfffffffeu);   // the "no candidate" pattern never passes
        int mine = 0;
#pragma unroll
        for (int t = 0; t < 32; ++t) mine += db[t] <= thr ? 1 : 0;
        int incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int v = __shfl_up_sync(0xffffffffu, incl, o);
          if (lane >= o) incl += v;
        }
        const int c = __shfl_sync(0xffffffffu, incl, 31);
        if (c == 0) continue;           // warp-uniform
        if (c <= 64) {
          uint2* slot = myq + (incl - mine);
          const unsigned idx0 = (unsigned)(base + sub + lane * 4);
#pragma unroll
          for (int t = 0; t < 32; ++t) {
            if (db[t] <= thr) *slot++ = make_uint2(db[t], idx0 + (unsigned)((t >> 2) * 128 + (t & 3)));
          }
          __syncwarp();
          int o = 0;
          if (first && sub == 0 && c >= 32) {   // nothing selected yet: the sorted first 32 entries are the list
            const uint2 e = myq[lane];
            const uint2 r = knn_sort_call(e.x, e.y, kmask);
            td = r.x;
            ti = r.y;
            o = 32;
          }
          if (c - o > 12) {
            for (; o < c; o += 32) {
              const uint2 e = o + lane < c ? myq[o + lane] : make_uint2(0xffffffffu, 0xffffffffu);
              knn_merge(td, ti, e.x, e.y, lane, kmask);
            }
          } else {
#pragma unroll 1
            for (; o < c; ++o) {
              const uint2 e = myq[o];
              knn_insert(td, ti, e.x, e.y, lane);
            }
          }
          tau = __shfl_sync(0xffffffffu, td, 31);
          __syncwarp();                 // the queue is rewritten by the next sub-chunk / query
          continue;
        }
        // ---- incremental path: more than 64 candidates under the bound (ties)
        int qn = 0;
#pragma unroll 1
        for (int t = 0; t < 32; ++t) {
          unsigned dt = 0;               // db[t] without dynamic register indexing
#pragma unroll
          for (int u = 0; u < 32; ++u) dt = u == t ? db[u] : dt;
          const bool pass = dt <= thr;
          const unsigned m = __ballot_sync(0xffffffffu, pass);
          if (m == 0u) continue;
          if (pass)
            myq[qn + __popc(m & lt_mask)] = make_uint2(dt, (unsigned)(base + sub + ((t >> 2) * 32 + lane) * 4 + (t & 3)));
          qn += __popc(m);
          __syncwarp();
          if (qn >= 32) {
            const uint2 e = myq[lane];
            knn_merge(td, ti, e.x, e.y, lane, kmask);
            tau = __shfl_sync(0xffffffffu, td, 31);
            thr = min(thr, tau);
            const int rem = qn - 32;
            const uint2 carry = lane < rem ? myq[32 + lane] : make_uint2(0u, 0u);
            __syncwarp();
            if (lane < rem) myq[lane] = carry;
            __syncwarp();
            qn = rem;
          }
        }
        if (qn > 0) {   // flush so that the next sub-chunk starts from an exact 32nd distance
          const uint2 e = lane < qn ? myq[lane] : make_uint2(0xffffffffu, 0xffffffffu);
          knn_merge(td, ti, e.x, e.y, lane, kmask);
          tau = __shfl_sync(0xffffffffu, td, 31);
          __syncwarp();
        }
      }
      if (!last) {
        park_d[warp][w][lane] = td;
        park_i[warp][w][lane] = ti;
      } else if (lane < K) {
        const size_t o = ((size_t)b * S + q) * K + lane;
        if (out64) out64[o] = (int64_t)ti;
        if (out_rows32) out_rows32[o] = b * N + (int)ti;
        if (out_d2) out_d2[o] = __uint_as_float(td);
      }
    }
  }
}

// ======================================================================================
// kNN for LARGE clouds (2048 < N <= KG_MAXN, the dataset shape 11000): block pruning.  The whole cloud is binned by
// the CTA into an 8 x 8 x 8 grid over its bounding box and laid out in shared memory in Morton order of the cells
// (histogram with one shared-memory atomic per point, a 512-entry scan, a cursor scatter), so that every run of 128
// consecutive points -- a BLOCK, which a warp scans with one float4 per lane and plane -- is a compact region with its
// own bounding box.  Per query the warp computes the distance to every block's box with the SAME rounded operations as
// the point distances (sqdist3 to the clamped query; every operation is monotonic, so the bound never exceeds the
// computed distance of a point inside), visits the blocks in ascending order of that bound and stops as soon as the
// smallest remaining bound exceeds the current 32nd distance.  Distances are still ((dx^2 + dy^2) + dz^2) with
// round-to-nearest multiplies and adds and the order is still (distance, ORIGINAL index): bit-identical to the exhaustive
// scan (pointnet_util.py:118-119), of which a 11000-point cloud visits ~5 %.  (For N <= 2048 the same scheme was measured
// SLOWER than the exhaustive kernel above -- 2080 vs 1328 warp instructions per query, profiles/r02_knn_block_pruning_
// experiment.txt -- and is not used there.)
// ======================================================================================
constexpr int KG_BLK = 128;                 // points per block
constexpr int KG_MAXN = 14336;              // 112 blocks: planes + permutation + boxes fit 227 KB
constexpr int KG_WARPS = 16;                // warps per CTA (one CTA per SM: the cloud fills its shared memory)
constexpr int KG_QPW = 8;                   // queries per warp (amortises binning the cloud)
constexpr int KG_PB = 8;                    // points per thread and batch of the binning passes (loads issued together)
#ifndef PZ_KG_BITS
#define PZ_KG_BITS 3
#endif
constexpr int KG_BITS = PZ_KG_BITS;          // grid cells per axis = 2^KG_BITS
constexpr int KG_CELLS = 1 << (3 * KG_BITS);
__device__ __forceinline__ unsigned fkey(float x) {   // order-preserving image of a float (for redux min / max)
  const unsigned b = __float_as_uint(x);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float fkey_inv(unsigned k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}
__device__ __forceinline__ int kg_cell(float x, float y, float z, const float (&lo)[3], const float (&inv)[3]) {
  constexpr int G = (1 << KG_BITS) - 1;
  const int ix = min(G, max(0, (int)((x - lo[0]) * inv[0])));
  const int iy = min(G, max(0, (int)((y - lo[1]) * inv[1])));
  const int iz = min(G, max(0, (int)((z - lo[2]) * inv[2])));
  int c = 0;   // Morton order: bit 3 b + {0, 1, 2} = bit b of {x, y, z}
#pragma unroll
  for (int b = 0; b < KG_BITS; ++b) c |= (((ix >> b) & 1) << (3 * b)) | (((iy >> b) & 1) << (3 * b + 1)) | (((iz >> b) & 1) << (3 * b + 2));
  return c;
}
// exclusive scan of the KG_CELLS cell counts in place (one warp, KG_CELLS / 32 consecutive counts per lane)
__device__ __forceinline__ void kg_scan(int* hist, int lane) {
  constexpr int PER = KG_CELLS / 32;
  int sum = 0;
  for (int j = 0; j < PER; ++j) sum += hist[lane * PER + j];
  int incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  int run = incl - sum;
  for (int j = 0; j < PER; ++j) {
    const int c = hist[lane * PER + j];
    hist[lane * PER + j] = run;
    run += c;
  }
}

__global__ void __launch_bounds__(KG_WARPS * 32, 1) knn_grid_kernel(const float* __restrict__ query,
                                                                     const float* __restrict__ xyz, int S, int N, int K,
                                                                     int64_t* __restrict__ out64,
                                                                     int* __restrict__ out_rows32,
                                                                     float* __restrict__ out_d2) {
  extern __shared__ __align__(16) unsigned char kg_smem[];
  const int nblk = (N + KG_BLK - 1) / KG_BLK, npad = nblk * KG_BLK, pstride = npad + 4;
  float* pts = reinterpret_cast<float*>(kg_smem);                              // x / y / z planes, sorted order
  unsigned short* perm = reinterpret_cast<unsigned short*>(pts + 3 * pstride); // sorted position -> original index
  float* bbox = reinterpret_cast<float*>(perm + npad);                         // [nblk][6]: lo xyz, hi xyz
  int* hist = reinterpret_cast<int*>(bbox + 6 * nblk);                         // [KG_CELLS]
  unsigned* redk = reinterpret_cast<unsigned*>(hist + KG_CELLS);               // [KG_WARPS][6]
  uint2* qkey = reinterpret_cast<uint2*>(redk + KG_WARPS * 6);                 // [KG_WARPS][64]
  const int b = blockIdx.y;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* p = xyz + (size_t)b * N * 3;
  const unsigned kmask = bitonic_keep_mask(lane);
  uint2* myq = qkey + warp * 64;
  const unsigned lt_mask = (1u << lane) - 1u;

  // ---- bounding box of the cloud
  unsigned kmin[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, kmax[3] = {0u, 0u, 0u};
  constexpr int T = KG_WARPS * 32;
  // every pass walks the cloud in batches of KG_PB points per thread whose 3 * KG_PB loads are issued together (the
  // shared-memory atomics of the later passes would otherwise serialise one global-memory latency per point)
  for (int base = tid; base < N; base += T * KG_PB) {
    float v[KG_PB][3];
#pragma unroll
    for (int u = 0; u < KG_PB; ++u) {
      const int i = min(base + u * T, N - 1);
#pragma unroll
      for (int d = 0; d < 3; ++d) v[u][d] = p[(size_t)i * 3 + d];
    }
#pragma unroll
    for (int u = 0; u < KG_PB; ++u) {
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        const unsigned kk = fkey(v[u][d]);
        kmin[d] = min(kmin[d], kk);
        kmax[d] = max(kmax[d], kk);
      }
    }
  }
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    const unsigned mn = __reduce_min_sync(0xffffffffu, kmin[d]), mx = __reduce_max_sync(0xffffffffu, kmax[d]);
    if (lane == 0) { redk[warp * 6 + d] = mn; redk[warp * 6 + 3 + d] = mx; }
  }
  for (int i = tid; i < KG_CELLS; i += T) hist[i] = 0;
  __syncthreads();
  float lo[3], inv[3];
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    unsigned mn = 0xffffffffu, mx = 0u;
#pragma unroll
    for (int w = 0; w < KG_WARPS; ++w) { mn = min(mn, redk[w * 6 + d]); mx = max(mx, redk[w * 6 + 3 + d]); }
    lo[d] = fkey_inv(mn);
    const float ext = fkey_inv(mx) - lo[d];
    inv[d] = ext > 0.f ? (float)(1 << KG_BITS) / ext : 0.f;
  }
  // ---- histogram of the cells, exclusive scan (cursor per cell), scatter in Morton order
  for (int base = tid; base < N; base += T * KG_PB) {
    float v[KG_PB][3];
#pragma unroll
    for (int u = 0; u < KG_PB; ++u) {
      const int i = min(base + u * T, N - 1);
#pragma unroll
      for (int d = 0; d < 3; ++d) v[u][d] = p[(size_t)i * 3 + d];
    }
#pragma unroll
    for (int u = 0; u < KG_PB; ++u)
      if (base + u * T < N) atomicAdd(&hist[kg_cell(v[u][0], v[u][1], v[u][2], lo, inv)], 1);
  }
  __syncthreads();
  if (warp == 0) {
    kg_scan(hist, lane);
  }
  __syncthreads();
  for (int base = tid; base < N; base += T * KG_PB) {
    float v[KG_PB][3];
#pragma unroll
    for (int u = 0; u < KG_PB; ++u) {
      const int i = min(base + u * T, N - 1);
#pragma unroll
      for (int d = 0; d < 3; ++d) v[u][d] = p[(size_t)i * 3 + d];
    }
#pragma unroll
    for (int u = 0; u < KG_PB; ++u) {
      const int i = base + u * T;
      if (i < N) {
        const int pos = atomicAdd(&hist[kg_cell(v[u][0], v[u][1], v[u][2], lo, inv)], 1);
        pts[pos] = v[u][0];
        pts[pstride + pos] = v[u][1];
        pts[2 * pstride + pos] = v[u][2];
        perm[pos] = (unsigned short)i;
      }
    }
  }
  // the tail of the last block: far-away points (distance ~3e36); their index (N + something) is never read (K <= N)
  for (int i = N + tid; i < npad; i += T) {
    pts[i] = pts[pstride + i] = pts[2 * pstride + i] = 1e18f;
    perm[i] = 0xffffu;
  }
  __syncthreads();
  for (int blk = warp; blk < nblk; blk += KG_WARPS) {   // bounding boxes of the blocks (real points only)
    const int i0 = blk * KG_BLK + lane * 4;
    unsigned bmin[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, bmax[3] = {0u, 0u, 0u};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (i0 + j < N) {
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          const unsigned k = fkey(pts[d * pstride + i0 + j]);
          bmin[d] = min(bmin[d], k);
          bmax[d] = max(bmax[d], k);
        }
      }
    }
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      const unsigned mn = __reduce_min_sync(0xffffffffu, bmin[d]), mx = __reduce_max_sync(0xffffffffu, bmax[d]);
      if (lane == 0) { bbox[blk * 6 + d] = fkey_inv(mn); bbox[blk * 6 + 3 + d] = fkey_inv(mx); }
    }
  }
  __syncthreads();

  // ---- queries
  const int q0 = (blockIdx.x * KG_WARPS + warp) * KG_QPW;
#pragma unroll 1
  for (int w = 0; w < KG_QPW; ++w) {
    const int q = q0 + w;
    if (q >= S) break;                  // warp-uniform
    const float* qp = query + ((size_t)b * S + q) * 3;
    const float qx = qp[0], qy = qp[1], qz = qp[2];
    unsigned td = 0xffffffffu, ti = 0xffffffffu;   // lane l holds the l-th smallest key so far
    unsigned tau = 0xffffffffu;                    // distance bits of the current 32nd smallest
    unsigned lbv[4];                               // lower bounds of blocks lane, lane + 32, lane + 64, lane + 96
#pragma unroll
    for (int sl = 0; sl < 4; ++sl) {
      const int blk = sl * 32 + lane;
      lbv[sl] = 0xffffffffu;
      if (blk < nblk) {
        const float cx = fminf(fmaxf(qx, bbox[blk * 6 + 0]), bbox[blk * 6 + 3]);
        const float cy = fminf(fmaxf(qy, bbox[blk * 6 + 1]), bbox[blk * 6 + 4]);
        const float cz = fminf(fmaxf(qz, bbox[blk * 6 + 2]), bbox[blk * 6 + 5]);
        lbv[sl] = min(__float_as_uint(sqdist3(qx, qy, qz, cx, cy, cz)), 0xfffffffeu);
      }
    }
#pragma unroll 1
    while (true) {
      const unsigned mine_lb = min(min(lbv[0], lbv[1]), min(lbv[2], lbv[3]));
      const unsigned mlb = __reduce_min_sync(0xffffffffu, mine_lb);
      if (mlb == 0xffffffffu || mlb > tau) break;   // every remaining point is farther than the 32nd
      const int src = __ffs(__ballot_sync(0xffffffffu, mine_lb == mlb)) - 1;
      int blk = 0;
      if (lane == src) {                // the owning lane takes its first slot with that bound and marks it visited
        const int sl = lbv[0] == mlb ? 0 : (lbv[1] == mlb ? 1 : (lbv[2] == mlb ? 2 : 3));
        blk = sl * 32 + lane;
#pragma unroll
        for (int u = 0; u < 4; ++u) lbv[u] = u == sl ? 0xffffffffu : lbv[u];
      }
      blk = __shfl_sync(0xffffffffu, blk, src);
      const int i0 = blk * KG_BLK + lane * 4;
      const float4 X = *reinterpret_cast<const float4*>(pts + i0);
      const float4 Y = *reinterpret_cast<const float4*>(pts + pstride + i0);
      const float4 Z = *reinterpret_cast<const float4*>(pts + 2 * pstride + i0);
      unsigned db[4];
      db[0] = __float_as_uint(sqdist3(qx, qy, qz, X.x, Y.x, Z.x));
      db[1] = __float_as_uint(sqdist3(qx, qy, qz, X.y, Y.y, Z.y));
      db[2] = __float_as_uint(sqdist3(qx, qy, qz, X.z, Y.z, Z.z));
      db[3] = __float_as_uint(sqdist3(qx, qy, qz, X.w, Y.w, Z.w));
      const bool have = tau != 0xffffffffu;
      unsigned thr = tau;
      if (!have) {                      // warp-uniform: nothing selected yet -> a bound from the lane minima
        const unsigned lo01 = min(db[0], db[1]), hi01 = max(db[0], db[1]), lo23 = min(db[2], db[3]), hi23 = max(db[2], db[3]);
        const unsigned m0 = min(lo01, lo23), m1 = min(max(lo01, lo23), min(hi01, hi23));
        unsigned hi = __reduce_max_sync(0xffffffffu, m0);   // >= 32 candidates are <= the largest lane minimum
        unsigned lo2 = __reduce_min_sync(0xffffffffu, m1);
        if (lo2 < hi) {
#pragma unroll 1
          for (int it = 0; it < 8 && lo2 < hi; ++it) {
            const unsigned mid = lo2 + ((hi - lo2) >> 1);
            const int c = __reduce_add_sync(0xffffffffu, (m0 <= mid ? 1 : 0) + (m1 <= mid ? 1 : 0));
            if (c >= 32) hi = mid; else lo2 = mid + 1;
          }
        }
        thr = hi;
      }
      thr = min(thr, 0xfffffffeu);
      const int mine = (db[0] <= thr) + (db[1] <= thr) + (db[2] <= thr) + (db[3] <= thr);
      int incl = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
      }
      const int c = __shfl_sync(0xffffffffu, incl, 31);
      if (c == 0) continue;             // warp-uniform
      const uint2 pm = *reinterpret_cast<const uint2*>(perm + i0);   // four 16-bit original indices
      const unsigned idx4[4] = {pm.x & 0xffffu, pm.x >> 16, pm.y & 0xffffu, pm.y >> 16};
      if (c <= 64) {
        uint2* slot = myq + (incl - mine);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          if (db[t] <= thr) *slot++ = make_uint2(db[t], idx4[t]);
        }
        __syncwarp();
        int o = 0;
        if (!have && c >= 32) {         // nothing selected yet: the sorted first 32 entries are the list
          const uint2 e = myq[lane];
          const uint2 r = knn_sort_call(e.x, e.y, kmask);
          td = r.x;
          ti = r.y;
          o = 32;
        }
        if (c - o > 12) {
          for (; o < c; o += 32) {
            const uint2 e = o + lane < c ? myq[o + lane] : make_uint2(0xffffffffu, 0xffffffffu);
            knn_merge(td, ti, e.x, e.y, lane, kmask);
          }
        } else {
#pragma unroll 1
          for (; o < c; ++o) {
            const uint2 e = myq[o];
            knn_insert(td, ti, e.x, e.y, lane);
          }
        }
        tau = __shfl_sync(0xffffffffu, td, 31);
        __syncwarp();                   // the queue is rewritten by the next block / query
        continue;
      }
      // ---- more than 64 candidates under the bound (ties, the padded block): 32 at a time through the merge network
      int qn = 0;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const bool pass = db[t] <= thr;
        const unsigned m = __ballot_sync(0xffffffffu, pass);
        if (m == 0u) continue;
        if (pass) myq[qn + __popc(m & lt_mask)] = make_uint2(db[t], idx4[t]);
        qn += __popc(m);
        __syncwarp();
        if (qn >= 32) {
          const uint2 e = myq[lane];
          knn_merge(td, ti, e.x, e.y, lane, kmask);
          tau = __shfl_sync(0xffffffffu, td, 31);
          thr = min(thr, tau);
          const int rem = qn - 32;
          const uint2 carry = lane < rem ? myq[32 + lane] : make_uint2(0u, 0u);
          __syncwarp();
          if (lane < rem) myq[lane] = carry;
          __syncwarp();
          qn = rem;
        }
      }
      if (qn > 0) {
        const uint2 e = lane < qn ? myq[lane] : make_uint2(0xffffffffu, 0xffffffffu);
        knn_merge(td, ti, e.x, e.y, lane, kmask);
        __syncwarp();
      }
      tau = __shfl_sync(0xffffffffu, td, 31);
    }
    if (lane < K) {
      const size_t o = ((size_t)b * S + q) * K + lane;
      if (out64) out64[o] = (int64_t)ti;
      if (out_rows32) out_rows32[o] = b * N + (int)ti;
      if (out_d2) out_d2[o] = __uint_as_float(td);
    }
  }
}

// ======================================================================================
// FPS for LARGE clouds (4096 < N <= KG_MAXN) with block-pruned updates.  The exhaustive kernels above touch all N
// running minima in every one of the S iterations; here the cloud is binned and Morton-ordered once (as in
// knn_grid_kernel), every 128-point block keeps its current maximum of the running minima, and an iteration only
// updates the blocks the new centroid can reach: a block is skipped when the distance from the centroid to its bounding
// box -- computed with the same rounded operations as the point distances, so it never exceeds any of them -- is >= the
// block's maximum (then fminf(md, d) = md for every point inside).  After a few dozen samples most blocks are skipped.
// The selection is unchanged: arg-max of the running minima, lowest ORIGINAL index on ties (pointnet_util.py:67-72), so
// the sampled indices are bit-identical.  One CTA of 16 warps per cloud; warp w owns blocks w, w + 16, ...: their running
// minima live in registers (4 points per lane and block), lane j < 8 carries the box, the maximum and the arg-max key of
// the warp's j-th block; per iteration one ballot finds the blocks to update, two redux give the warp's best key, one
// CTA barrier and two more redux the winner.
// ======================================================================================
constexpr int FG_WARPS = 16, FG_T = FG_WARPS * 32, FG_SLOTS = 8;   // FG_SLOTS blocks per warp: KG_MAXN / 128 / 16 = 7
__global__ void __launch_bounds__(FG_T, 1) fps_grid_kernel(const float* __restrict__ xyz, int N, int S,
                                                           const int64_t* __restrict__ start, int64_t* __restrict__ out64,
                                                           int* __restrict__ out_rows32, float* __restrict__ new_xyz) {
  extern __shared__ __align__(16) unsigned char fg_smem[];
  const int nblk = (N + KG_BLK - 1) / KG_BLK, npad = nblk * KG_BLK, pstride = npad + 4;
  float* pts = reinterpret_cast<float*>(fg_smem);                              // x / y / z planes, Morton order
  unsigned short* perm = reinterpret_cast<unsigned short*>(pts + 3 * pstride); // sorted position -> original index
  float* bbox = reinterpret_cast<float*>(perm + npad);                         // [nblk][6]
  int* hist = reinterpret_cast<int*>(bbox + 6 * nblk);                         // [KG_CELLS]
  unsigned* redk = reinterpret_cast<unsigned*>(hist + KG_CELLS);               // [FG_WARPS][6]
  unsigned* wkey = redk + FG_WARPS * 6;                                        // [2 parities][FG_WARPS][2] (hi, lo)
  int* sel = reinterpret_cast<int*>(wkey + 2 * FG_WARPS * 2);                  // [S] picked original indices
  const int c = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* p = xyz + (size_t)c * N * 3;
  constexpr int T = FG_T;

  // ---- bin the cloud (see knn_grid_kernel): bounding box, histogram of the 8 x 8 x 8 cells, scan, scatter
  unsigned kmin[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, kmax[3] = {0u, 0u, 0u};
  for (int base = tid; base < N; base += T * KG_PB) {
    float v[KG_PB][3];
#pragma unroll
    for (int u = 0; u < KG_PB; ++u) {
      const int i = min(base + u * T, N - 1);
#pragma unroll
      for (int d = 0; d < 3; ++d) v[u][d] = p[(size_t)i * 3 + d];
    }
#pragma unroll
    for (int u = 0; u < KG_PB; ++u) {
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        const unsigned kk = fkey(v[u][d]);
        kmin[d] = min(kmin[d], kk);
        kmax[d] = max(kmax[d], kk);
      }
    }
  }
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    const unsigned mn = __reduce_min_sync(0xffffffffu, kmin[d]), mx = __reduce_max_sync(0xffffffffu, kmax[d]);
    if (lane == 0) { redk[warp * 6 + d] = mn; redk[warp * 6 + 3 + d] = mx; }
  }
  for (int i = tid; i < KG_CELLS; i += T) hist[i] = 0;
  if (tid < 2 * FG_WARPS * 2) wkey[tid] = 0u;
  __syncthreads();
  float lo[3], inv[3];
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    unsigned mn = 0xffffffffu, mx = 0u;
#pragma unroll
    for (int w = 0; w < FG_WARPS; ++w) { mn = min(mn, redk[w * 6 + d]); mx = max(mx, redk[w * 6 + 3 + d]); }
    lo[d] = fkey_inv(mn);
    const float ext = fkey_inv(mx) - lo[d];
    inv[d] = ext > 0.f ? (float)(1 << KG_BITS) / ext : 0.f;
  }
  for (int base = tid; base < N; base += T * KG_PB) {
    float v[KG_PB][3];
#pragma unroll
    for (int u = 0; u < KG_PB; ++u) {
      const int i = min(base + u * T, N - 1);
#pragma unroll
      for (int d = 0; d < 3; ++d) v[u][d] = p[(size_t)i * 3 + d];
    }
#pragma unroll
    for (int u = 0; u < KG_PB; ++u)
      if (base + u * T < N) atomicAdd(&hist[kg_cell(v[u][0], v[u][1], v[u][2], lo, inv)], 1);
  }
  __syncthreads();
  if (warp == 0) {
    kg_scan(hist, lane);
  }
  __syncthreads();
  for (int base = tid; base < N; base += T * KG_PB) {
    float v[KG_PB][3];
#pragma unroll
    for (int u = 0; u < KG_PB; ++u) {
      const int i = min(base + u * T, N - 1);
#pragma unroll
      for (int d = 0; d < 3; ++d) v[u][d] = p[(size_t)i * 3 + d];
    }
#pragma unroll
    for (int u = 0; u < KG_PB; ++u) {
      const int i = base + u * T;
      if (i < N) {
        const int pos = atomicAdd(&hist[kg_cell(v[u][0], v[u][1], v[u][2], lo, inv)], 1);
        pts[pos] = v[u][0];
        pts[pstride + pos] = v[u][1];
        pts[2 * pstride + pos] = v[u][2];
        perm[pos] = (unsigned short)i;
      }
    }
  }
  for (int i = N + tid; i < npad; i += T) {      // padding of the last block: never selected (running minimum 0, largest index)
    pts[i] = pts[pstride + i] = pts[2 * pstride + i] = 0.f;
    perm[i] = 0xffffu;
  }
  __syncthreads();
  for (int blk = warp; blk < nblk; blk += FG_WARPS) {   // bounding boxes of the blocks (real points only)
    const int i0 = blk * KG_BLK + lane * 4;
    unsigned bmin[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, bmx[3] = {0u, 0u, 0u};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (i0 + j < N) {
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          const unsigned k = fkey(pts[d * pstride + i0 + j]);
          bmin[d] = min(bmin[d], k);
          bmx[d] = max(bmx[d], k);
        }
      }
    }
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      const unsigned mn = __reduce_min_sync(0xffffffffu, bmin[d]), mx = __reduce_max_sync(0xffffffffu, bmx[d]);
      if (lane == 0) { bbox[blk * 6 + d] = fkey_inv(mn); bbox[blk * 6 + 3 + d] = fkey_inv(mx); }
    }
  }
  __syncthreads();

  // ---- per-warp state: running minima of the owned blocks (registers), lane j < FG_SLOTS: box / maximum / key of block j
  float md[FG_SLOTS][4];
#pragma unroll
  for (int j = 0; j < FG_SLOTS; ++j) {
    const int i0 = (warp + FG_WARPS * j) * KG_BLK + lane * 4;
#pragma unroll
    for (int i = 0; i < 4; ++i) md[j][i] = (warp + FG_WARPS * j < nblk && i0 + i < N) ? 1e10f : 0.f;
  }
  const int myblk = warp + FG_WARPS * lane;                  // the block lane `lane` speaks for (lanes < FG_SLOTS)
  const bool owns = lane < FG_SLOTS && myblk < nblk;
  float bb[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (owns) {
#pragma unroll
    for (int d = 0; d < 6; ++d) bb[d] = bbox[myblk * 6 + d];
  }
  unsigned bmax = owns ? __float_as_uint(1e10f) : 0u, blo = 0u;   // block maximum (bits) and its key (~original index | position)

  int far = (int)start[c];
  far = min(max(far, 0), N - 1);
  float cx = p[(size_t)far * 3], cy = p[(size_t)far * 3 + 1], cz = p[(size_t)far * 3 + 2];
  for (int s = 0; s < S; ++s) {
    if (tid == 0) sel[s] = far;
    if (s + 1 == S) break;
    // which of my blocks can the new centroid change?  (the distance to the box never exceeds a point's distance)
    bool need = false;
    if (owns) {
      const float qx = fminf(fmaxf(cx, bb[0]), bb[3]), qy = fminf(fmaxf(cy, bb[1]), bb[4]), qz = fminf(fmaxf(cz, bb[2]), bb[5]);
      need = __float_as_uint(sqdist3(qx, qy, qz, cx, cy, cz)) < bmax;
    }
    const unsigned needmask = __ballot_sync(0xffffffffu, need);
#pragma unroll
    for (int j = 0; j < FG_SLOTS; ++j) {
      if ((needmask >> j) & 1u) {                            // warp-uniform
        const int i0 = (warp + FG_WARPS * j) * KG_BLK + lane * 4;
        const float4 X = *reinterpret_cast<const float4*>(pts + i0);
        const float4 Y = *reinterpret_cast<const float4*>(pts + pstride + i0);
        const float4 Z = *reinterpret_cast<const float4*>(pts + 2 * pstride + i0);
        const uint2 pm = *reinterpret_cast<const uint2*>(perm + i0);
        md[j][0] = fminf(md[j][0], sqdist3(X.x, Y.x, Z.x, cx, cy, cz));
        md[j][1] = fminf(md[j][1], sqdist3(X.y, Y.y, Z.y, cx, cy, cz));
        md[j][2] = fminf(md[j][2], sqdist3(X.z, Y.z, Z.z, cx, cy, cz));
        md[j][3] = fminf(md[j][3], sqdist3(X.w, Y.w, Z.w, cx, cy, cz));
        // key = (running minimum bits, ~original index << 16 | sorted position): largest minimum, lowest original index
        const unsigned l0 = ((0xffffu - (pm.x & 0xffffu)) << 16) | (unsigned)i0, l1 = ((0xffffu - (pm.x >> 16)) << 16) | (unsigned)(i0 + 1);
        const unsigned l2 = ((0xffffu - (pm.y & 0xffffu)) << 16) | (unsigned)(i0 + 2), l3 = ((0xffffu - (pm.y >> 16)) << 16) | (unsigned)(i0 + 3);
        unsigned hi = __float_as_uint(md[j][0]), lo2 = l0;
        { const unsigned h = __float_as_uint(md[j][1]); const bool g = h > hi || (h == hi && l1 > lo2); hi = g ? h : hi; lo2 = g ? l1 : lo2; }
        { const unsigned h = __float_as_uint(md[j][2]); const bool g = h > hi || (h == hi && l2 > lo2); hi = g ? h : hi; lo2 = g ? l2 : lo2; }
        { const unsigned h = __float_as_uint(md[j][3]); const bool g = h > hi || (h == hi && l3 > lo2); hi = g ? h : hi; lo2 = g ? l3 : lo2; }
        const unsigned mhi = __reduce_max_sync(0xffffffffu, hi);
        const unsigned mlo = __reduce_max_sync(0xffffffffu, hi == mhi ? lo2 : 0u);
        if (lane == j) { bmax = mhi; blo = mlo; }
      }
    }
    // the warp's best block, then the CTA's
    const unsigned whi = __reduce_max_sync(0xffffffffu, owns ? bmax : 0u);
    const unsigned wlo = __reduce_max_sync(0xffffffffu, (owns && bmax == whi) ? blo : 0u);
    const int par = s & 1;
    if (lane == 0) {
      wkey[(par * FG_WARPS + warp) * 2] = whi;
      wkey[(par * FG_WARPS + warp) * 2 + 1] = wlo;
    }
    __syncthreads();
    const unsigned h2 = lane < FG_WARPS ? wkey[(par * FG_WARPS + lane) * 2] : 0u;
    const unsigned l2k = lane < FG_WARPS ? wkey[(par * FG_WARPS + lane) * 2 + 1] : 0u;
    const unsigned ghi = __reduce_max_sync(0xffffffffu, h2);
    const unsigned glo = __reduce_max_sync(0xffffffffu, h2 == ghi ? l2k : 0u);
    const int pos = (int)(glo & 0xffffu);
    far = (int)(0xffffu - (glo >> 16));
    cx = pts[pos]; cy = pts[pstride + pos]; cz = pts[2 * pstride + pos];
  }
  __syncthreads();
  for (int s = tid; s < S; s += T) {
    const int f = sel[s];
    const size_t o = (size_t)c * S + s;
    if (out64) out64[o] = f;
    if (out_rows32) out_rows32[o] = c * N + f;
    if (new_xyz) {
      new_xyz[o * 3 + 0] = p[(size_t)f * 3];
      new_xyz[o * 3 + 1] = p[(size_t)f * 3 + 1];
      new_xyz[o * 3 + 2] = p[(size_t)f * 3 + 2];
    }
  }
}

static int fps_grid_launch(const float* xyz, int B, int N, const int64_t* start, int S, int64_t* out64, int* out_rows32,
                           float* new_xyz, cudaStream_t st) {
  const int nblk = (N + KG_BLK - 1) / KG_BLK, npad = nblk * KG_BLK;
  PZ_REQUIRE(nblk <= FG_WARPS * FG_SLOTS, PZ_ERR_UNSUPPORTED, "pz_fps: N=%d exceeds the block-pruned kernel's %d points", N, FG_WARPS * FG_SLOTS * KG_BLK);
  const size_t smem = (size_t)3 * (npad + 4) * sizeof(float) + (size_t)npad * sizeof(unsigned short) + (size_t)6 * nblk * sizeof(float) +
                      KG_CELLS * sizeof(int) + FG_WARPS * 6 * sizeof(unsigned) + 2 * FG_WARPS * 2 * sizeof(unsigned) + (size_t)S * sizeof(int);
  PZ_REQUIRE(smem <= 232448, PZ_ERR_UNSUPPORTED, "pz_fps: N=%d, S=%d need %zu B of shared memory", N, S, smem);
  PZ_CUDA(cudaFuncSetAttribute(fps_grid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  fps_grid_kernel<<<B, FG_T, smem, st>>>(xyz, N, S, start, out64, out_rows32, new_xyz);
  PZ_LAUNCH_CHECK();
  return 0;
}

int launch_knn(const float* query, const float* xyz, int B, int S, int N, int K, int64_t* out64,
               int* out_rows32, float* out_d2, cudaStream_t st) {
  PZ_REQUIRE(K >= 1 && K <= 32, PZ_ERR_UNSUPPORTED, "pz_knn: K=%d not in [1,32]", K);
  PZ_REQUIRE(N >= K, PZ_ERR_UNSUPPORTED, "pz_knn: N=%d < K=%d", N, K);
  PZ_REQUIRE(B <= 65535, PZ_ERR_UNSUPPORTED, "pz_knn: B=%d > 65535", B);
  if (N > KNN_CHUNK && N <= KG_MAXN && S >= 64) {        // large clouds (the dataset shape): block pruning
    const int nblk = (N + KG_BLK - 1) / KG_BLK, npad = nblk * KG_BLK;
    const size_t smem = (size_t)3 * (npad + 4) * sizeof(float) + (size_t)npad * sizeof(unsigned short) + (size_t)6 * nblk * sizeof(float) +
                        KG_CELLS * sizeof(int) + KG_WARPS * 6 * sizeof(unsigned) + (size_t)KG_WARPS * 64 * sizeof(uint2);
    PZ_REQUIRE(smem <= 232448, PZ_ERR_UNSUPPORTED, "pz_knn: N=%d needs %zu B of shared memory", N, smem);
    PZ_CUDA(cudaFuncSetAttribute(knn_grid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((S + KG_WARPS * KG_QPW - 1) / (KG_WARPS * KG_QPW), B);
    knn_grid_kernel<<<grid, KG_WARPS * 32, smem, st>>>(query, xyz, S, N, K, out64, out_rows32, out_d2);
    PZ_LAUNCH_CHECK();
    return 0;
  }
  dim3 grid((S + KNN_WARPS * KNN_QPW - 1) / (KNN_WARPS * KNN_QPW), B);
  PZ_CUDA(launch_pdl(knn_kernel, grid, dim3(KNN_WARPS * 32), 0, st, query, xyz, S, N, K, out64, out_rows32, out_d2));
  PZ_LAUNCH_CHECK();
  return 0;
}

// ======================================================================================
// square_distance (materialising API): HBM-write bound, 128-bit stores along N.
// ======================================================================================
__global__ void __launch_bounds__(256) sqdist_kernel(const float* __restrict__ src,
                                                     const float* __restrict__ dst, int S, int N,
                                                     float* __restrict__ out) {
  const int b = blockIdx.z;
  const int s = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (s >= S) return;
  const float* sp = src + ((size_t)b * S + s) * 3;
  const float sx = sp[0], sy = sp[1], sz = sp[2];
  const float* dp = dst + (size_t)b * N * 3;
  float* op = out + ((size_t)b * S + s) * N;
  const int lane = threadIdx.x & 31;
  for (int n = blockIdx.x * 32 * 4 + lane; n < N; n += gridDim.x * 32 * 4) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      int i = n + u * 32;
      if (i < N) op[i] = sqdist3(sx, sy, sz, dp[i * 3 + 0], dp[i * 3 + 1], dp[i * 3 + 2]);
    }
  }
}

// ======================================================================================
// ball query: one thread per query scans the cloud in index order (pointnet_util.py:76-96)
// ======================================================================================
__global__ void __launch_bounds__(128) ball_query_kernel(const float* __restrict__ xyz,
                                                         const float* __restrict__ new_xyz, int N,
                                                         int S, float r2, int nsample,
                                                         int64_t* __restrict__ out) {
  const int b = blockIdx.y;
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  const float* qp = new_xyz + ((size_t)b * S + s) * 3;
  const float qx = qp[0], qy = qp[1], qz = qp[2];
  const float* p = xyz + (size_t)b * N * 3;
  int64_t* o = out + ((size_t)b * S + s) * nsample;
  int cnt = 0;
  int64_t first = N;
  for (int i = 0; i < N && cnt < nsample; ++i) {
    float d = sqdist3(qx, qy, qz, p[i * 3], p[i * 3 + 1], p[i * 3 + 2]);
    if (!(d > r2)) {
      if (cnt == 0) first = i;
      o[cnt++] = i;
    }
  }
  for (; cnt < nsample; ++cnt) o[cnt] = first;
}

// ======================================================================================
// index_points: generic row gather in 4-byte or 1-byte units
// ======================================================================================
template <typename U>
__global__ void __launch_bounds__(256) gather_rows_kernel(const U* __restrict__ pts,
                                                          const int64_t* __restrict__ idx, int N,
                                                          int row_units, int M, size_t total,
                                                          U* __restrict__ out) {
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total;
       e += (size_t)gridDim.x * blockDim.x) {
    size_t row = e / row_units;
    int u = (int)(e - row * row_units);
    size_t b = row / M;
    int64_t j = idx[row];
    out[e] = pts[(b * N + (size_t)j) * row_units + u];
  }
}

// ======================================================================================
// grouping tail of sample_and_group: new_points[b,s,k,:] = [xyz[j]-ctr, feat[j]]
// ======================================================================================
__global__ void __launch_bounds__(256) group_concat_kernel(const float* __restrict__ xyz,
                                                           const float* __restrict__ feat,
                                                           const float* __restrict__ new_xyz,
                                                           const int64_t* __restrict__ knn, int N,
                                                           int D, int S, int K, size_t rows, int ld,
                                                           float* __restrict__ new_points,
                                                           float* __restrict__ grouped_xyz) {
  const int W = ld;                                // row stride >= 3 + D; the columns beyond 3 + D are zero-filled
  const int lane = threadIdx.x & 31;
  const size_t warp0 = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const size_t nwarps = ((size_t)gridDim.x * blockDim.x) >> 5;
  for (size_t r = warp0; r < rows; r += nwarps) {  // r = (b*S + s)*K + k
    const size_t bs = r / K;
    const size_t b = bs / S;
    const size_t j = b * N + (size_t)knn[r];
    float* o = new_points + r * W;
    if (lane < 3) {
      float v = xyz[j * 3 + lane];
      o[lane] = __fsub_rn(v, new_xyz[bs * 3 + lane]);
      if (grouped_xyz) grouped_xyz[r * 3 + lane] = v;
    }
    for (int d = lane; d < D; d += 32) o[3 + d] = feat[j * D + d];
    for (int d = 3 + D + lane; d < W; d += 32) o[d] = 0.f;
  }
}

// ------------------------------------------------------------------ plane_split (dataset.py:761-775)
// Order-preserving two-way partition of clouds by the sign of  p . normal + z  (evaluated in float64, as numpy does
// for a float32 cloud and a float64 normal).  One CTA per cloud walks it in chunks of 1024 points: ballot + warp
// counts + a scan over the 32 warps give every point its slot in `up` (dis >= 0) or `down` (dis < 0).  With
// pad != 0 the unused tail rows of both outputs are filled with copies of their first row (FPS-safe padding).
__global__ void __launch_bounds__(1024) plane_split_kernel(const float* __restrict__ pts_all, const int* __restrict__ sizes,
                                                           int n_stride, int C, const double* __restrict__ planes,
                                                           float* __restrict__ up_all, float* __restrict__ down_all,
                                                           int* __restrict__ counts, int pad) {
  __shared__ int warp_up[32], warp_dn[32];
  __shared__ int base_up, base_dn;
  const int piece = blockIdx.x;
  const int n = sizes ? sizes[piece] : n_stride;
  const float* pts = pts_all + (size_t)piece * n_stride * C;
  float* up = up_all + (size_t)piece * n_stride * C;
  float* down = down_all + (size_t)piece * n_stride * C;
  const double nx = planes[piece * 4], ny = planes[piece * 4 + 1], nz = planes[piece * 4 + 2], z = planes[piece * 4 + 3];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  if (t == 0) { base_up = 0; base_dn = 0; }
  __syncthreads();
  for (int c0 = 0; c0 < n; c0 += 1024) {
    const int i = c0 + t;
    bool valid = i < n, is_up = false;
    if (valid) {
      const float* p = pts + (size_t)i * C;
      const double dis = ((double)p[0] * nx + (double)p[1] * ny) + (double)p[2] * nz + z;
      is_up = dis >= 0.0;
    }
    const unsigned mu = __ballot_sync(0xffffffffu, valid && is_up), md = __ballot_sync(0xffffffffu, valid && !is_up);
    if (lane == 0) { warp_up[warp] = __popc(mu); warp_dn[warp] = __popc(md); }
    __syncthreads();
    int off_u = base_up, off_d = base_dn;
    for (int w = 0; w < warp; ++w) { off_u += warp_up[w]; off_d += warp_dn[w]; }
    if (valid) {
      const unsigned lt = (1u << lane) - 1u;
      float* dst = is_up ? up + (size_t)(off_u + __popc(mu & lt)) * C : down + (size_t)(off_d + __popc(md & lt)) * C;
      const float* p = pts + (size_t)i * C;
      for (int c = 0; c < C; ++c) dst[c] = p[c];
    }
    __syncthreads();
    if (t == 0) {
      int su = 0, sd = 0;
      for (int w = 0; w < 32; ++w) { su += warp_up[w]; sd += warp_dn[w]; }
      base_up += su;
      base_dn += sd;
    }
    __syncthreads();
  }
  if (t == 0) { counts[piece * 2] = base_up; counts[piece * 2 + 1] = base_dn; }
  if (pad) {
    const int nu = base_up, nd = base_dn;
    for (int e = nu * C + t; e < n_stride * C; e += 1024) up[e] = nu > 0 ? up[e % C] : 0.f;
    for (int e = nd * C + t; e < n_stride * C; e += 1024) down[e] = nd > 0 ? down[e % C] : 0.f;
  }
}

}  // namespace pz

// ------------------------------------------------------------------------- C ABI
using namespace pz;

extern "C" int pz_plane_split(const float* pts, const int32_t* sizes_or_null, int P, int n_stride, int C,
                              const double* planes, float* up, float* down, int32_t* counts, int pad_tail,
                              pz_stream_t stream) {
  PZ_REQUIRE(P >= 0 && n_stride >= 0 && C >= 3, PZ_ERR_ARG, "pz_plane_split: need P, n >= 0 and at least 3 columns (C=%d)", C);
  if (P == 0) return 0;
  PZ_REQUIRE(planes && counts && (n_stride == 0 || (pts && up && down)), PZ_ERR_ARG, "pz_plane_split: null pointer");
  plane_split_kernel<<<P, 1024, 0, as_stream(stream)>>>(pts, sizes_or_null, n_stride, C, planes, up, down, counts, pad_tail);
  PZ_LAUNCH_CHECK();
  return 0;
}

extern "C" int pz_fps(const float* xyz, int B, int N, const int64_t* start, int S, int64_t* out_idx,
                      float* new_xyz_or_null, pz_stream_t stream) {
  PZ_REQUIRE(B >= 0 && N >= 1 && S >= 1, PZ_ERR_ARG, "pz_fps: bad sizes B=%d N=%d S=%d", B, N, S);
  if (B == 0) return 0;
  PZ_REQUIRE(xyz && start && out_idx, PZ_ERR_ARG, "pz_fps: null pointer");
  return launch_fps(xyz, B, N, start, S, out_idx, nullptr, new_xyz_or_null, as_stream(stream));
}

extern "C" int pz_knn(const float* query, const float* xyz, int B, int S, int N, int K,
                      int64_t* out_idx, float* out_d2_or_null, pz_stream_t stream) {
  PZ_REQUIRE(B >= 0 && S >= 0 && N >= 1, PZ_ERR_ARG, "pz_knn: bad sizes B=%d S=%d N=%d", B, S, N);
  if (B == 0 || S == 0) return 0;
  PZ_REQUIRE(query && xyz && out_idx, PZ_ERR_ARG, "pz_knn: null pointer");
  return launch_knn(query, xyz, B, S, N, K, out_idx, nullptr, out_d2_or_null, as_stream(stream));
}

extern "C" int pz_sqdist(const float* src, const float* dst, int B, int S, int N, float* out,
                         pz_stream_t stream) {
  PZ_REQUIRE(B >= 0 && S >= 0 && N >= 0, PZ_ERR_ARG, "pz_sqdist: bad sizes");
  if (B == 0 || S == 0 || N == 0) return 0;
  PZ_REQUIRE(src && dst && out, PZ_ERR_ARG, "pz_sqdist: null pointer");
  PZ_REQUIRE(B <= 65535 && (S + 7) / 8 <= 65535, PZ_ERR_UNSUPPORTED, "pz_sqdist: grid too large");
  int gx = (N + 127) / 128;
  if (gx > 64) gx = 64;
  dim3 grid(gx, (S + 7) / 8, B);
  sqdist_kernel<<<grid, 256, 0, as_stream(stream)>>>(src, dst, S, N, out);
  PZ_LAUNCH_CHECK();
  return 0;
}

extern "C" int pz_ball_query(const float* xyz, const float* new_xyz, int B, int N, int S,
                             float radius, int nsample, int64_t* out_idx, pz_stream_t stream) {
  PZ_REQUIRE(B >= 0 && N >= 1 && S >= 0 && nsample >= 1, PZ_ERR_ARG, "pz_ball_query: bad sizes");
  if (B == 0 || S == 0) return 0;
  PZ_REQUIRE(xyz && new_xyz && out_idx, PZ_ERR_ARG, "pz_ball_query: null pointer");
  PZ_REQUIRE(B <= 65535, PZ_ERR_UNSUPPORTED, "pz_ball_query: B > 65535");
  dim3 grid((S + 127) / 128, B);
  ball_query_kernel<<<grid, 128, 0, as_stream(stream)>>>(xyz, new_xyz, N, S, radius * radius, nsample, out_idx);
  PZ_LAUNCH_CHECK();
  return 0;
}

extern "C" int pz_gather(const void* pts, const int64_t* idx, int B, int N, int C, int M,
                         int elem_bytes, void* out, pz_stream_t stream) {
  PZ_REQUIRE(B >= 0 && N >= 1 && C >= 1 && M >= 0 && elem_bytes >= 1, PZ_ERR_ARG, "pz_gather: bad sizes");
  if (B == 0 || M == 0) return 0;
  PZ_REQUIRE(pts && idx && out, PZ_ERR_ARG, "pz_gather: null pointer");
  size_t row_bytes = (size_t)C * elem_bytes;
  bool words = (row_bytes % 4 == 0) && ((uintptr_t)pts % 4 == 0) && ((uintptr_t)out % 4 == 0);
  size_t unit = words ? 4 : 1;
  int row_units = (int)(row_bytes / unit);
  size_t total = (size_t)B * M * row_units;
  int blocks = (int)((total + 255) / 256 < (size_t)kNumSMs * 16 ? (total + 255) / 256 : (size_t)kNumSMs * 16);
  if (words)
    gather_rows_kernel<uint32_t><<<blocks, 256, 0, as_stream(stream)>>>((const uint32_t*)pts, idx, N, row_units, M, total, (uint32_t*)out);
  else
    gather_rows_kernel<uint8_t><<<blocks, 256, 0, as_stream(stream)>>>((const uint8_t*)pts, idx, N, row_units, M, total, (uint8_t*)out);
  PZ_LAUNCH_CHECK();
  return 0;
}

// The HBM-bound form of the same op (SURVEY.md 8d: the materialising sample_and_group API is a pure gather + write of
// 4*S*K*(3+D) bytes per cloud): ONE WARP PER GROUP.  The K = 32 gathered rows of a group are one contiguous run of
// 32*(3+D) floats in the output, so the warp assembles the run in shared memory (feature rows arrive as fully coalesced
// 16-byte loads, two rows per warp instruction; the three centred coordinates per row from lane k) and writes it out as
// 16-byte stores over the contiguous run -- the run starts on a 16-byte boundary because 32*(3+D)*4 is a multiple of 16.
// Needs K == 32 and D % 4 == 0 (the model's shapes); everything else takes group_concat_kernel above.
template <int WARPS, int D4>
__global__ void __launch_bounds__(WARPS * 32) group_concat_tile_kernel(const float* __restrict__ xyz, const float* __restrict__ feat,
                                                                        const float* __restrict__ new_xyz,
                                                                        const int64_t* __restrict__ knn, int N, int D, int S,
                                                                        size_t groups, float* __restrict__ new_points,
                                                                        float* __restrict__ grouped_xyz) {
  extern __shared__ __align__(16) float gc_smem[];
  const int W = 3 + D, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* tile = gc_smem + (size_t)warp * 32 * W;              // [32][W], 32*W*4 bytes: a multiple of 16
  const int d4 = D >> 2;                                       // float4 pieces per feature row
  for (size_t g = (size_t)blockIdx.x * WARPS + warp; g < groups; g += (size_t)gridDim.x * WARPS) {
    const size_t b = g / S;
    const size_t r0 = g * 32;
    const size_t jl = b * N + (size_t)knn[r0 + lane];          // lane k owns neighbour k's source row
    {                                                          // centred coordinates (pointnet_util.py:125)
      const float cx = new_xyz[g * 3], cy = new_xyz[g * 3 + 1], cz = new_xyz[g * 3 + 2];
      const float x = xyz[jl * 3], y = xyz[jl * 3 + 1], z = xyz[jl * 3 + 2];
      tile[lane * W] = __fsub_rn(x, cx);
      tile[lane * W + 1] = __fsub_rn(y, cy);
      tile[lane * W + 2] = __fsub_rn(z, cz);
      if (grouped_xyz) {
        grouped_xyz[(r0 + lane) * 3] = x;
        grouped_xyz[(r0 + lane) * 3 + 1] = y;
        grouped_xyz[(r0 + lane) * 3 + 2] = z;
      }
    }
    // features: piece p = (row p / d4, float4 p % d4); consecutive lanes read consecutive 16 bytes of a row.  All loads
    // of a batch of pieces are issued before the first is stored (the gather is latency bound otherwise).
    if (D4 > 0) {                                              // compile-time D: every load of the group in flight at once
      float4 v[D4 > 0 ? D4 : 1];
#pragma unroll
      for (int i = 0; i < D4; ++i) {
        const int p = lane + 32 * i, k = p / D4, c = p % D4;
        const size_t j = __shfl_sync(0xffffffffu, jl, k);
        v[i] = __ldg(reinterpret_cast<const float4*>(feat + j * D) + c);
      }
#pragma unroll
      for (int i = 0; i < D4; ++i) {
        const int p = lane + 32 * i, k = p / D4, c = p % D4;
        float* t = tile + k * W + 3 + c * 4;
        t[0] = v[i].x; t[1] = v[i].y; t[2] = v[i].z; t[3] = v[i].w;
      }
    } else {
      for (int p = lane; p < 32 * d4; p += 32) {
        const int k = p / d4, c = p - k * d4;
        const size_t j = __shfl_sync(0xffffffffu, jl, k);
        const float4 v = __ldg(reinterpret_cast<const float4*>(feat + j * D) + c);
        float* t = tile + k * W + 3 + c * 4;
        t[0] = v.x; t[1] = v.y; t[2] = v.z; t[3] = v.w;
      }
    }
    __syncwarp();
    float4* dst = reinterpret_cast<float4*>(new_points + r0 * W);
    const float4* src = reinterpret_cast<const float4*>(tile);
    for (int p = lane; p < 8 * W; p += 32) dst[p] = src[p];   // 32*W floats = 8*W float4
    __syncwarp();
  }
}

extern "C" int pz_group_concat(const float* xyz, const float* feat_or_null, const float* new_xyz,
                               const int64_t* knn_idx, int B, int N, int D, int S, int K,
                               float* new_points, float* grouped_xyz_or_null, pz_stream_t stream) {
  PZ_REQUIRE(B >= 0 && N >= 1 && D >= 0 && S >= 0 && K >= 1, PZ_ERR_ARG, "pz_group_concat: bad sizes");
  const int ld = 3 + D;
  size_t rows = (size_t)B * S * K;
  if (rows == 0) return 0;
  PZ_REQUIRE(xyz && new_xyz && knn_idx && new_points, PZ_ERR_ARG, "pz_group_concat: null pointer");
  PZ_REQUIRE(feat_or_null || D == 0, PZ_ERR_ARG, "pz_group_concat: feat is null but D=%d", D);
  if (K == 32 && D >= 4 && D % 4 == 0 && D <= 256 && ((uintptr_t)feat_or_null & 15) == 0 && ((uintptr_t)new_points & 15) == 0) {
    constexpr int WARPS = 4;
    const size_t groups = (size_t)B * S;
    const size_t smem = (size_t)WARPS * 32 * ld * sizeof(float);
    const size_t want_t = (groups + WARPS - 1) / WARPS;
    const int blocks_t = (int)(want_t < (size_t)kNumSMs * 8 ? want_t : (size_t)kNumSMs * 8);
    auto launch = [&](auto kern) {
      PZ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      kern<<<blocks_t, WARPS * 32, smem, as_stream(stream)>>>(xyz, feat_or_null, new_xyz, knn_idx, N, D, S, groups, new_points,
                                                              grouped_xyz_or_null);
      return 0;
    };
    if (D == 64) PZ_TRY(launch(group_concat_tile_kernel<WARPS, 16>));         // the model's stage 1 / the C3 shape
    else if (D == 128) PZ_TRY(launch(group_concat_tile_kernel<WARPS, 32>));   // the model's stage 2
    else PZ_TRY(launch(group_concat_tile_kernel<WARPS, 0>));
    PZ_LAUNCH_CHECK();
    return 0;
  }
  size_t want = (rows + 7) / 8;
  int blocks = (int)(want < (size_t)kNumSMs * 16 ? want : (size_t)kNumSMs * 16);
  group_concat_kernel<<<blocks, 256, 0, as_stream(stream)>>>(xyz, feat_or_null, new_xyz, knn_idx, N, D, S, K, rows, ld, new_points, grouped_xyz_or_null);
  PZ_LAUNCH_CHECK();
  return 0;
}
