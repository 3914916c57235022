// Shared helpers for libpuzzlenet_sm100.so (internal; the public ABI is include/puzzlenet_b200.h).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <utility>

#include "../../include/puzzlenet_b200.h"

namespace pz {

// thread-local last-error text behind pz_last_error()
char* error_buffer();
int fail(int code, const char* fmt, ...);

#define PZ_REQUIRE(cond, code, ...)                      \
  do {                                                   \
    if (!(cond)) return ::pz::fail((code), __VA_ARGS__); \
  } while (0)

#define PZ_CUDA(expr)                                                                   \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess)                                                              \
      return ::pz::fail((int)_e, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                        __FILE__, __LINE__);                                            \
  } while (0)

// every kernel launch site is followed by exactly one PZ_LAUNCH_CHECK(): it also feeds pz_launch_count()
#define PZ_LAUNCH_CHECK()            \
  do {                               \
    ::pz::count_launch();            \
    PZ_CUDA(cudaGetLastError());     \
  } while (0)

// Programmatic dependent launch (PDL) of the forward's kernel chain.  A kernel launched through launch_pdl() may become
// resident while its predecessor in the stream is still draining (launch latency, barrier / TMEM set-up and descriptor
// fetches overlap the predecessor's tail); every such kernel calls pdl_enter() BEFORE its first access to global memory:
// it blocks until the predecessor grid has completed and its writes are visible, and only then lets the successor in, so
// at most two grids of the chain are in flight and a resident CTA never runs ahead of anything but its direct predecessor.
// Only kernels that call pdl_enter() may be launched with launch_pdl().
// Measured (B=64 split forward, 1 B200): eager launches on one stream 1.59 -> 1.51 ms per forward.  NOT used under stream
// capture: in the 4-stream graph schedule the early-resident CTAs of one stream's next kernel hold SMs that another
// stream's ready kernel would have used (1.37 -> 1.52 ms per step), nor with the stage recorder on (an event record between
// two launches turns the programmatic edge into a slower full one: 1.67 -> 1.79 ms).
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_enter() {
  pdl_wait();
  pdl_trigger();
}
#endif
bool pdl_for_stream(cudaStream_t st);   // capi.cu: the stage recorder is off and `st` is not capturing
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_for_stream(st) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

// propagate a non-zero status from an internal call
#define PZ_TRY(expr)         \
  do {                       \
    int _s = (expr);         \
    if (_s != 0) return _s;  \
  } while (0)

void count_launch();
// opt-in stage profiler (pz_profile_*): CUDA events between the stages of pz_predict5 / pz_encoder_forward
void prof_begin(cudaStream_t st);
void prof_mark(const char* stage, cudaStream_t st, int lane = 0);   // lane 1 = the internal side stream

// Internal fork/join helper: one non-blocking side stream + events per (device, caller stream), created on first use
// and reused by every call on that stream (capturable: the side stream is always joined back into the caller's stream).
struct SideStream {
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, join_a = nullptr, join_b = nullptr;
};
int side_stream(SideStream** out, cudaStream_t caller);
bool prof_serial();   // pz_profile_enable(2): run the geometry chain on the caller's stream (clean per-stage times)

static inline cudaStream_t as_stream(pz_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// bump allocator over the caller's workspace
struct Arena {
  char* base;
  size_t size;
  size_t used;
  Arena(void* p, size_t n) : base(static_cast<char*>(p)), size(n), used(0) {}
  template <typename T>
  T* take(size_t count) {
    size_t off = align_up(used, 256);
    used = off + count * sizeof(T);
    return reinterpret_cast<T*>(base + off);
  }
  bool ok() const { return used <= size; }
};

constexpr int kNumSMs = 148;  // B200

// ---- internal launchers shared between translation units -------------------------------

// fps.cu / knn.cu: int32 "global row" outputs feed the fused grouping kernels.
int launch_fps(const float* xyz, int B, int N, const int64_t* start64, int S, int64_t* out64,
               int* out_rows32, float* new_xyz, cudaStream_t st);
int launch_knn(const float* query, const float* xyz, int B, int S, int N, int K, int64_t* out64,
               int* out_rows32, float* out_d2, cudaStream_t st);

// gemm_f32.cu
struct GemmF32 {
  // Y[M,N] = epilogue(A[M,K] * W[N,K]^T + bias[N]); all row-major, K contiguous.
  const float* A = nullptr;
  int lda = 0;
  const float* W[2] = {nullptr, nullptr};  // weight set w = row / rows_per_wset
  const float* bias[2] = {nullptr, nullptr};
  int ldw = 0;
  int rows_per_wset = 0;  // 0 -> single set
  float* Y = nullptr;
  int ldy = 0;
  int M = 0, N = 0, K = 0;
  int relu = 0;
  float alpha = 1.f;  // applied to the accumulator before bias
  int ksplit = 0;     // >0: split K over grid.z in chunks of ksplit, raw partials to Y + z*M*ldy
  // EPI_RESIDUAL: Y = R + relu(acc + bias)
  const float* R = nullptr;
  int ldr = 0;
  // EPI_ROWBIAS: extra per-row-block bias table rb[(row / rb_rows), N]
  const float* rowbias = nullptr;
  int rb_rows = 0;
  // EPI_GROUPMAX: Y[M/G, N] = relu?(max over G consecutive rows + bias); G in {32, 128}
  int group = 0;
  // gathered A (grouped-MLP layer 2): A[r,k] = relu(F[rows[r],k] + b1[k] + W1x[k,:] . (xyz[rows[r]] - ctr[r/32]))
  const int* rows = nullptr;      // [M] global row ids into F / xyz
  const float* xyz = nullptr;     // [*,3]
  const float* centers = nullptr; // [M/32,3]
  const float* W1[2] = {nullptr, nullptr};  // [K, ldw1] first three columns used
  const float* b1[2] = {nullptr, nullptr};  // [K]
  int ldw1 = 0;
};
int launch_gemm_f32(const GemmF32& g, cudaStream_t st);

// gemm_tc.cu -- tcgen05 bf16 GEMM: D^T[ch,row] = W[ch,:] . X[row,:]  (see the file header)
long long* kernel_timeline_buffer(long long min_slots);   // pz_profile_attention_timeline's buffer if it holds >= min_slots int64, else null
struct TcGemm {
  long long* prof = nullptr;                       // gather mode: CTA 0 stamps its first jobs (slots 1024.., 1280.., 1408..)
  const __nv_bfloat16* W[2] = {nullptr, nullptr};  // [Nout, K] bf16 row-major, weight set = row / rows_per_wset
  int ldw = 0;
  const float* bias[2] = {nullptr, nullptr};       // [Nout] fp32
  int rows_per_wset = 0;
  const __nv_bfloat16* X = nullptr;                // plain: activations [M, K]; gathered: P [*, K]
  int ldx = 0;
  const int* rows = nullptr;                       // gathered: source row of P for each of the M rows
  const float* centers = nullptr;                  // gathered: [M/32, 3] fp32 group centres; X[r] = relu(P[rows[r]] - Q[r/32])
                                                   //   with Q[g,k] = W1x[k,0:3] . centers[g] computed per stage in smem
  int M = 0, Nout = 0, K = 0;
  int epi = 0;                                     // 0 store rows, 1 max over groups of 32 rows, 2 max over the tile's rows
  int relu = 0;
  float* Yf = nullptr;                             // fp32 output (optional)
  int ldyf = 0;
  __nv_bfloat16* Yb = nullptr;                     // bf16 output (optional)
  int ldyb = 0;
  const float* Rf = nullptr;                       // residual added after the ReLU (fp32 or bf16 source)
  int ldrf = 0;
  const __nv_bfloat16* Rb = nullptr;
  int ldrb = 0;
  int n_valid = 0;                                 // >0: only channels < n_valid exist (weights zero-padded to Nout)
  const float* rowbias = nullptr;                  // epi 0: + rowbias[(row / rb_rows) * rb_ld + ch] before the ReLU
  int rb_rows = 0, rb_ld = 0;
  float* Ymax = nullptr;                           // epi 0: also Ymax[tile * ldmax + ch] = max over the tile's rows
  int ldmax = 0;
  __nv_bfloat16* YT = nullptr;                     // split row GEMM: output stored TRANSPOSED per block of t_rows rows
  const float* xyz = nullptr;                      // epi 0 only: y += W1x[ch,0:3] . xyz[row]  (layer 1 of a grouped MLP)
  const float* W1x[2] = {nullptr, nullptr};
  int ldw1x = 0;
  // ---- split path (gemm_split.cu): every 16-bit tensor is a pair of fp16 planes, hi (the pointer above) and lo (below),
  // with the same leading dimension
  const __nv_bfloat16* Xlo = nullptr;
  const __nv_bfloat16* Wlo[2] = {nullptr, nullptr};
  __nv_bfloat16* Yblo = nullptr;
  const __nv_bfloat16* Rblo = nullptr;
  __nv_bfloat16* YTlo = nullptr;
  int t_rows = 0;                                  // split row GEMM: rows per transposed block (YT), e.g. 256 = one cloud
  const float* Xf = nullptr;                       // split gather: P [*, K] fp32 (row stride ldx)
  const float* Qf = nullptr;                       // split gather: Q [M/32, K] fp32 = W1x[:, 0:3] . centre
};
int launch_tc_gemm(const TcGemm& g, cudaStream_t st);
// gemm_split.cu -- the same products as three fp16 MMAs (hi*hi + hi*lo + lo*hi), fp32 accumulation (PZ_PREC_SPLIT)
int launch_split_rowgemm(const TcGemm& g, cudaStream_t st);
int launch_split_gather(const TcGemm& g, cudaStream_t st);
int launch_split_planes(const float* in, size_t ldi, size_t rows, int cols, void* hi, void* lo, size_t ldo, cudaStream_t st);
// attention_split.cu: per cloud  r = x - softmax(q k^T / sqrt(64)) v  with split operands; q|k planes [rows,128],
// v^T planes [cloud][256 ch][256 tokens], x / r planes (ldx / 256)
struct AttnSplit {
  const void *qk_hi = nullptr, *qk_lo = nullptr, *vT_hi = nullptr, *vT_lo = nullptr, *x_hi = nullptr, *x_lo = nullptr;
  int ldx = 0;
  void *r_hi = nullptr, *r_lo = nullptr;
  float* attn = nullptr;
  int attn_mode = 0;
  // fused out-projection (wo_hi[0] != null): instead of r the kernel writes  out = x + relu(Wo r + bo)  as planes y (and as
  // fp32 rows yf when given); Wo planes [256, 256] fp16 K-major and bo [256] per weight set, cloud / clouds_per_set = set
  const void *wo_hi[2] = {nullptr, nullptr}, *wo_lo[2] = {nullptr, nullptr};
  const float* bo[2] = {nullptr, nullptr};
  int clouds_per_set = 0;
  void *y_hi = nullptr, *y_lo = nullptr;
  int ldy = 0;
  float* yf = nullptr;
  int ldyf = 0;
  // chained projections (wqkv_hi[0] != null; needs the fused out-projection): the kernel also computes the NEXT layer's
  // [q | k | v] = out Wqkv^T + b from its output rows (they never leave the SM between the two products) and writes the next
  // layer's q|k planes [rows, 128] and v^T planes [cloud][256 ch][256 tokens] -- into buffers other than qk / vT, which the
  // other CTAs of this launch are still reading.  Wqkv planes [384, 256] fp16 K-major and bias [384] per weight set.
  const void *wqkv_hi[2] = {nullptr, nullptr}, *wqkv_lo[2] = {nullptr, nullptr};
  const float* bqkv[2] = {nullptr, nullptr};
  void *qk2_hi = nullptr, *qk2_lo = nullptr, *vT2_hi = nullptr, *vT2_lo = nullptr;
  // cloud-granular hand-over between consecutive chained launches (256 CTAs on 148 SMs = 1.73 waves each: the second wave
  // of a layer leaves 40 SMs idle).  sig_flags[cloud] is incremented by each of a cloud's two CTAs after their last store;
  // a launch with dep_flags set is started with programmatic stream serialisation (its CTAs become resident as soon as every
  // CTA of the previous launch is) and every CTA waits for dep_flags[cloud] == 2 instead of the whole previous grid.
  const int* dep_flags = nullptr;
  int* sig_flags = nullptr;
};
int launch_attention_split(const AttnSplit& p, int clouds, cudaStream_t st);
// heads_split.cu: the boundary heads of predict5 as split-fp16 chained-MMA kernels (used by the split and bf16 paths)
struct HeadMlp3 {
  const float *w0, *b0, *w1, *b1, *w2, *b2;
};
constexpr size_t HEAD_SPLIT_IMG_SET = (size_t)(2 * 3 * 64 + 2 * (64 + 32)) * 72;   // fp16 elements of one set's weight images
int launch_heads_split(const float* xfeat, const HeadMlp3& pre_f, const HeadMlp3& pre_r, const HeadMlp3& seg_f,
                       const HeadMlp3& seg_r, int B, bool reuse_images, void* img, float* local, float* tilemax,
                       float* de_fpcb, float* de_mrpcb, cudaStream_t st);
int launch_seg_pairs_split(const HeadMlp3& pre_f, const HeadMlp3& pre_r, const HeadMlp3& seg_f, const HeadMlp3& seg_r,
                           bool reuse_images, void* img, const float* local_fpc, const float* tilemax_mrpc,
                           const int64_t* pairs, int n, float* de_fpcb, cudaStream_t st);
int launch_tc_rowgemm(const TcGemm& g, cudaStream_t st);   // gemm_tc_rows.cu: same struct, row-major store epilogue
// attention_layer_tc.cu: a stack of 1-4 offset-attention layers per cloud in ONE launch (per layer: projections, softmax,
// P v, out-proj, residuals); layer l + 1 reads the output of layer l
struct AttnLayerTc {
  int nlayers = 1;
  const __nv_bfloat16* x = nullptr;       // [clouds*256, ldx] input of layer 0
  int ldx = 0;
  // per layer 20 pre-swizzled [128 x 64] tile images (16 KB each): Wqkv [384, 256] (q rows 0-63, k 64-127, v 128-383) as
  // tiles (row block, k-block) 0-11, then Wo [256, 256] as tiles 12-19 (launch_attn_weight_image); layers contiguous
  const __nv_bfloat16* wimg[2] = {nullptr, nullptr};
  const float* bqkv[2] = {nullptr, nullptr};           // [nlayers][384]
  const float* bo[2][4] = {{nullptr, nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr, nullptr}};   // [256] per layer
  int clouds_per_set = 0;
  __nv_bfloat16* yb = nullptr;            // [clouds*256, ldyb] output of layer 0; layer l at yb + l * yb_layer_stride
  int ldyb = 0;
  size_t yb_layer_stride = 0;
  float* yf = nullptr;                    // optional fp32 copy, layer l at yf + l * yf_layer_stride
  int ldyf = 0;
  size_t yf_layer_stride = 0;
  float* attn = nullptr;                  // attention map accumulation, mode per layer: 0 none, 1 store, 2 add,
                                          // 3 (sum + map) / 4 (the mean of the four layers' maps)
  int attn_mode[4] = {0, 0, 0, 0};
  long long* prof = nullptr;              // pz_profile_attention_timeline
};
int launch_attention_layer_tc(const AttnLayerTc& p, int clouds, cudaStream_t st);
constexpr size_t ATTN_WIMG_ELEMS = 20 * 128 * 64;   // bf16 elements of one layer's tile images
// fp32 rows [rows, 256] of a weight block -> their place in the tile images (row_off = first row inside the block
// sequence: q 0, k 64, v 128, o 384)
int launch_attn_weight_image(const float* src, int rows, int row_off, __nv_bfloat16* img, cudaStream_t st);
int launch_cvt_bf16(const float* in, int ldi, int rows, int cols, __nv_bfloat16* out, int ldo, cudaStream_t st);

}  // namespace pz
