/*
 * puzzlenet_b200.h -- C ABI of libpuzzlenet_sm100.so
 *
 * B200 (sm_100a) implementation of the PuzzleNet point-cloud encoder +
 * pair-matching forward and the approximate-EMD loss.  The reference is pure
 * Python/torch on this path; its "FFI" is the Python module boundary
 * (pointnet_util.*, model5_b.TouchedRegraster.predict5) plus one pybind11
 * module, emd_cuda (PyTorchEMD/cuda/emd.cpp:23-27).  Every entry point below
 * names the reference interface it replaces (paths relative to the reference
 * root).  INTEGRATION.md shows the ctypes binding the Python shims use.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host;
 *   - tensors are dense row-major fp32, indices are int64 at this boundary
 *     (the reference returns torch.long);
 *   - nothing is allocated inside: scratch comes from the caller through a
 *     workspace pointer sized by the matching *_workspace_bytes() call;
 *   - every call is asynchronous on `stream` (a cudaStream_t), re-entrant and
 *     CUDA-graph capturable; no global state except the last-error string;
 *   - return value: 0 = ok, <0 = argument error (PZ_ERR_*), >0 = cudaError_t.
 *     pz_last_error() returns a thread-local description of the last failure.
 */
#ifndef PUZZLENET_B200_H_
#define PUZZLENET_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* pz_stream_t; /* cudaStream_t */

#define PZ_OK 0
#define PZ_ERR_ARG (-1)         /* null pointer / non-positive size / bad enum */
#define PZ_ERR_UNSUPPORTED (-2) /* size outside the supported range (see each call) */
#define PZ_ERR_WORKSPACE (-3)   /* workspace too small */

#define PZ_PREC_FP32 0 /* fp32 CUDA-core math, matches the reference to ~1e-6 rel */
#define PZ_PREC_BF16 1 /* bf16 operands, fp32 accumulate on tcgen05 tensor cores */
#define PZ_PREC_SPLIT 2 /* every operand as an fp16 hi/lo pair, three tcgen05 MMAs per product (hi*hi + hi*lo + lo*hi),
                         * fp32 accumulate: the tensor-core path that meets the fp32 tolerances (1e-4, 0.01 deg) */

#define PZ_ABI_VERSION 7

/* pz_predict5 flags */
#define PZ_FLAG_NEED 1          /* also return x2 / attention of both clouds (predict5 need=True) */
#define PZ_FLAG_REUSE_PACKS 2   /* the bf16 weight packs inside `workspace` are still valid: same workspace, same
                                   precision and unchanged weights since the previous call (skips one repack launch) */

int pz_abi_version(void);
const char* pz_last_error(void);
/* compute capability major*10+minor of the current device (100 on B200), <0 on error */
int pz_device_arch(void);

/* Instrumentation used by bench.py (the only process-global state besides the error string).
 * pz_launch_count: kernels launched by this library in this process so far.
 * pz_profile_enable(2): as 1, and the internal side stream is not used (stages run back to back on the caller's
 * stream), which gives per-stage times free of overlap.  While the recorder is on (1 or 2) the split precision launches
 * its kernels plainly instead of by programmatic dependent launch (an event between two launches would turn the
 * programmatic edge into a slower full one), so a recorded call is slower than an unrecorded one.
 * pz_profile_enable(1): record CUDA events on the caller's stream between the stages of every following
 * pz_predict5 / pz_encoder_forward call (at most 512 calls are kept); pz_profile_collect synchronises the
 * device, sums the elapsed milliseconds per stage over those calls into ms[0..n), stores the stage names
 * (static strings) and the number of profiled calls, resets the recorder and returns n. */
long long pz_launch_count(void);
int pz_profile_enable(int on);
int pz_profile_collect(double* ms_host, const char** names_host, int* calls_host, int max_stages);
/* Kernel-internal timelines: while a device buffer of n_slots int64 is registered, CTA 0 of every fused attention-layer
 * launch (attention_layer_tc.cu) stores SM clock stamps of its phase boundaries there (slots 0-17: epilogue thread 0,
 * 32-41: the MMA-issuing thread) and every CTA c its %globaltimer at entry / exit (64 + 2c, 65 + 2c) -- only when
 * n_slots >= 64 + 2 * clouds; CTA 0 of the stage-1 gather GEMM (gemm_tc.cu) stamps slots 1024..1455 -- only when
 * n_slots >= 1456.  Split path (%globaltimer, ns): the first CTA pair of the row GEMM launch selected by the environment
 * variable PZ_RG_TIMELINE (p1 | qk | vt | outproj | tail) stamps slots 2048..3071 (n_slots >= 3072), CTA 0 of every
 * attention_split_kernel launch slots 3072..3087 (n_slots >= 3088); scripts/rowgemm_timeline.py prints both.
 * A buffer too short for a stamp set switches that set off; n_slots < 64 is an argument error.
 * NULL switches everything off (the default). */
int pz_profile_attention_timeline(long long* device_buf_or_null, long long n_slots);

/* ---------------------------------------------------------------- geometry */

/* farthest_point_sample(xyz, npoint) -- pointnet_util.py:53-73.
 * xyz [B,N,3]; start [B] = the first centroid of each cloud (the reference draws it with
 * torch.randint on the CPU generator, pointnet_util.py:65 -- the caller does that draw);
 * out_idx [B,S].  Distances are ((dx*dx)+(dy*dy))+(dz*dz) in fp32 without FMA, argmax ties
 * resolve to the lowest index: bit-exact with the reference's CPU result.
 * new_xyz_or_null [B,S,3] receives xyz[out_idx] (index_points, pointnet_util.py:115).
 * Supported: 1 <= N <= 16384, 1 <= S. */
int pz_fps(const float* xyz, int B, int N, const int64_t* start, int S, int64_t* out_idx,
           float* new_xyz_or_null, pz_stream_t stream);

/* square_distance(src, dst) -- pointnet_util.py:22-36.  src [B,S,3], dst [B,N,3] -> out [B,S,N]. */
int pz_sqdist(const float* src, const float* dst, int B, int S, int N, float* out,
              pz_stream_t stream);

/* kNN selection = square_distance(query, xyz).argsort()[:, :, :K] -- pointnet_util.py:118-119,
 * without materialising [B,S,N].  query [B,S,3], xyz [B,N,3] -> out_idx [B,S,K] ascending by
 * (distance, index) (the reference's order among equal distances is undefined);
 * out_d2_or_null [B,S,K] the squared distances.  Supported: 1 <= K <= 32, N >= K. */
int pz_knn(const float* query, const float* xyz, int B, int S, int N, int K, int64_t* out_idx,
           float* out_d2_or_null, pz_stream_t stream);

/* query_ball_point(radius, nsample, xyz, new_xyz) -- pointnet_util.py:76-96.
 * First `nsample` indices (ascending) with d2 <= radius^2, padded with the first one; a query
 * with no point in range yields N everywhere, as the reference does. */
int pz_ball_query(const float* xyz, const float* new_xyz, int B, int N, int S, float radius,
                  int nsample, int64_t* out_idx, pz_stream_t stream);

/* index_points(points, idx) -- pointnet_util.py:39-50.  pts [B,N,C] of elem_bytes-sized
 * elements, idx [B,M] -> out [B,M,C].  Indices must lie in [0,N). */
int pz_gather(const void* pts, const int64_t* idx, int B, int N, int C, int M, int elem_bytes,
              void* out, pz_stream_t stream);

/* the grouping tail of sample_and_group -- pointnet_util.py:123-130.
 * new_points[b,s,k,:] = cat(xyz[b,knn[b,s,k]] - new_xyz[b,s], feat[b,knn[b,s,k]]) ([B,S,K,3+D]);
 * feat may be null (D = 0); grouped_xyz_or_null [B,S,K,3] = xyz[b,knn[b,s,k]] (returnfps=True). */
int pz_group_concat(const float* xyz, const float* feat_or_null, const float* new_xyz,
                    const int64_t* knn_idx, int B, int N, int D, int S, int K, float* new_points,
                    float* grouped_xyz_or_null, pz_stream_t stream);

/* plane_split(points, z) -- dataset.py:761-775, batched: P clouds stored [P, n_stride, C] (xyz first; cloud i has
 * sizes[i] valid rows, all n_stride when sizes is null) are each partitioned, order preserved, by the sign of
 * p . normal_i + z_i evaluated in float64 like numpy; planes [P,4] = (normal, z) as doubles ON THE DEVICE (the caller
 * draws them: np.random in the reference).  up (dis >= 0) / down (dis < 0) are [P, n_stride, C], counts [P,2].
 * pad_tail != 0 fills the unused rows with copies of the half's first row (safe padding for pz_fps). */
int pz_plane_split(const float* pts, const int32_t* sizes_or_null, int P, int n_stride, int C, const double* planes,
                   float* up, float* down, int32_t* counts, int pad_tail, pz_stream_t stream);

/* ------------------------------------------------------------ fused blocks */

/* sample_and_group's grouping + the shared MLP + neighbourhood max-pool in one pass, never
 * materialising [B,S,K,3+D]: model5_b.py:449-454 / :456-461 with pointnet_util.py:123-130.
 *   out[b,s,:] = max_k relu(W2 relu(W1 [xyz[j]-new_xyz[b,s] ; feat[j]] + b1) + b2),  j = knn[b,s,k]
 * W1 [C1,3+D], W2 [C2,C1] row-major (nn.Linear layout), K must be 32; B*S*K and B*N at most INT_MAX.
 * workspace: pz_group_mlp_workspace_bytes(B,N,D,S,K,C1,C2). */
size_t pz_group_mlp_workspace_bytes(int B, int N, int D, int S, int K, int C1, int C2);
int pz_group_mlp_maxpool(const float* xyz, const float* feat, const float* new_xyz,
                         const int64_t* knn_idx, const float* W1, const float* b1,
                         const float* W2, const float* b2, int B, int N, int D, int S, int K,
                         int C1, int C2, int precision, float* out, void* workspace,
                         size_t workspace_bytes, pz_stream_t stream);

/* nn.Linear on this path (every mlpN, out and tfMLP layer of model5_b.py): y = act(x W^T + b) (+ residual).
 * x [M,K] (row stride ldx), W [N,K], b [N] or null, residual_or_null [M,N] (row stride ldr) added
 * AFTER the optional ReLU (model5_b.py:100), y [M,N] (row stride ldy). */
int pz_linear(const float* x, int ldx, const float* W, const float* b, int M, int N, int K, int relu,
              const float* residual_or_null, int ldr, float* y, int ldy, int precision,
              pz_stream_t stream);

/* The same layer on the tcgen05 tensor cores with operands the caller already holds in bf16:
 * x_bf16 [M,K] (row stride ldx, elements), w_bf16 [N,K]; fp32 accumulate, fp32 bias/residual/output.
 * Supported: M % 256 == 0, N % 128 == 0, K % 64 == 0, 16-byte aligned rows. */
int pz_linear_bf16(const void* x_bf16, int ldx, const void* w_bf16, const float* b, int M, int N, int K,
                   int relu, const float* residual_or_null, int ldr, float* y, int ldy,
                   pz_stream_t stream);

/* layerAttention.forward -- model5_b.py:92-101.  x [B,L,C] -> out [B,L,C] = x + relu(Wo (x - A v) + bo),
 * attention_or_null [B,L,L].  Wq,Wk [C/4,C]; Wv,Wo [C,C].  Supported: C == 256, L as pz_scaled_dot_attention.
 * workspace: pz_offset_attention_workspace_bytes(B,L,C). */
size_t pz_offset_attention_workspace_bytes(int B, int L, int C);
int pz_offset_attention(const float* x, const float* Wq, const float* bq, const float* Wk,
                        const float* bk, const float* Wv, const float* bv, const float* Wo,
                        const float* bo, int B, int L, int C, int precision, float* out,
                        float* attention_or_null, void* workspace, size_t workspace_bytes,
                        pz_stream_t stream);

/* scaled_dot_production(q,k,v) -- model5_b.py:67-75 (mask=None).
 * q,k [B,L,Dk], v [B,L,Dv] -> values [B,L,Dv], attention_or_null [B,L,L].
 * Supported: L % 64 == 0, L <= 256, Dk == 64, Dv % 128 == 0. */
int pz_scaled_dot_attention(const float* q, const float* k, const float* v, int B, int L, int Dk,
                            int Dv, float* values, float* attention_or_null, pz_stream_t stream);

/* Parameters of one PCTransformer_nonsort (model5_b.py:417-441), nn.Linear layout
 * (weight [out,in] row-major, bias [out]); BatchNorm1d(1024) tensors are [1024]. */
typedef struct PzEncoderWeights {
  const float *mlp1_w, *mlp1_b; /* [64,3]    */
  const float *mlp2_w, *mlp2_b; /* [64,64]   */
  const float *mlp3_w, *mlp3_b; /* [128,67]  */
  const float *mlp4_w, *mlp4_b; /* [128,128] */
  const float *mlp5_w, *mlp5_b; /* [256,131] */
  const float *mlp6_w, *mlp6_b; /* [256,256] */
  const float *bn1_w, *bn1_b, *bn1_mean, *bn1_var;
  const float *bn2_w, *bn2_b, *bn2_mean, *bn2_var;
  const float *q_w[4], *q_b[4]; /* atten{1..4}.mlpq [64,256]  */
  const float *k_w[4], *k_b[4]; /* atten{1..4}.mlpk [64,256]  */
  const float *v_w[4], *v_b[4]; /* atten{1..4}.mlpv [256,256] */
  const float *o_w[4], *o_b[4]; /* atten{1..4}.out  [256,256] */
  const float *out_w, *out_b;   /* [1024,1280] */
} PzEncoderWeights;

/* Outputs of PCTransformer_nonsort.forward (model5_b.py:478) for E*B clouds; any pointer may be
 * null to skip that output (predict5 with need=False only consumes f_global and x_feature). */
typedef struct PzEncoderOutputs {
  float* f_global;  /* [E*B,1024]      */
  float* x2;        /* [E*B,256,3]     */
  float* attention; /* [E*B,256,256]   mean of the 4 maps (model5_b.py:468-469) */
  float* out;       /* [E*B,256,1024]  */
  float* x_feature; /* [E*B,1024,64]   */
  /* extra intermediates for parity tests (SURVEY.md Appendix A); null = skip */
  int64_t* fps1;    /* [E*B,512]       */
  int64_t* knn1;    /* [E*B,512,32]    */
  float* f1f;       /* [E*B,512,128]   */
  int64_t* fps2;    /* [E*B,256]       */
  int64_t* knn2;    /* [E*B,256,32]    */
  float* f2f;       /* [E*B,256,256]   */
  float* att_cat;   /* [E*B,256,1280]  cat(att1..att4, f2f) (model5_b.py:467,472) */
} PzEncoderOutputs;

/* Clouds per pz_encoder_forward call (E*B) and per pz_predict5 call (2B), in every precision: the kNN launches and the
 * fp32 attention put one cloud per grid row.  The test suite runs calls of up to 8190 clouds (pz_encode_pieces with
 * PZ_MAX_PIECES pieces, whose front half is pz_predict5's with B = P) and pz_predict5 up to B = 256. */
#define PZ_MAX_CLOUDS 65535

/* E encoders (different weight sets) over E*B clouds in one pass: cloud c uses weights[c / B].
 * xyz [E*B,1024,3]; start1 [E*B], start2 [E*B] = FPS start indices of stage 1 (in [0,1024)) and
 * stage 2 (in [0,512)).  Eval-mode BatchNorm (running statistics).  E in {1,2}.
 * Supported: 1 <= E*B <= PZ_MAX_CLOUDS (PZ_ERR_UNSUPPORTED otherwise, before any launch). */
size_t pz_encoder_workspace_bytes(int E, int B);
int pz_encoder_forward(const PzEncoderWeights* weights_host, int E, int B, const float* xyz,
                       const int64_t* start1, const int64_t* start2, int precision,
                       const PzEncoderOutputs* outputs_host, void* workspace,
                       size_t workspace_bytes, pz_stream_t stream);

/* Parameters of the pair heads (model5_b.py:561-599). */
typedef struct PzHeadWeights {
  const float *tf_w[5], *tf_b[5];         /* tfMLP.{0,2,4,6,8}: 2048-1024-512-512-256-6 */
  const float *pre_fpc_w[3], *pre_fpc_b[3]; /* MLPLocalPreFpc.{0,2,4} [64,64] */
  const float *pre_rpc_w[3], *pre_rpc_b[3]; /* MLPLocalPreRpc.{0,2,4} [64,64] */
  const float *seg_fpc_w[3], *seg_fpc_b[3]; /* MLPFpcb.{0,2,4}: 128-64-32-2 */
  const float *seg_rpc_w[3], *seg_rpc_b[3]; /* MLPRpcb.{0,2,4}: 128-64-32-2 */
} PzHeadWeights;

/* TouchedRegraster.predict5(batch, _, need, training=False) -- model5_b.py:672-759.
 * fpc, mrpc [B,1024,3]; starts [4,B] = FPS starts in the reference's draw order
 * (Encoder stage 1, Encoder stage 2, Encoder2 stage 1, Encoder2 stage 2; SURVEY.md App. A).
 * out6 [B,6]; de_fpcb, de_mrpcb [B,2,1024].  flags & PZ_FLAG_NEED additionally fills x2_* [B,256,3] and
 * attention_* [B,256,256] (may be null otherwise).  Reproduces the reference's use of the mrpc
 * global feature for both boundary heads (model5_b.py:741-744).
 * Supported: 1 <= B <= PZ_MAX_CLOUDS / 2 = 32767 (PZ_ERR_UNSUPPORTED otherwise, before any launch). */
size_t pz_predict5_workspace_bytes(int B);
int pz_predict5(const PzEncoderWeights* enc_host /*[2]*/, const PzHeadWeights* heads_host,
                const float* fpc, const float* mrpc, int B, const int64_t* starts, int precision,
                int flags, float* out6, float* de_fpcb, float* de_mrpcb, float* x2_fpc,
                float* attention_fpc, float* x2_mrpc, float* attention_mrpc, void* workspace,
                size_t workspace_bytes, pz_stream_t stream);

/* Pair scoring from per-piece encodings: pz_predict5 split at its pair boundary.  Everything pz_predict5 computes
 * before the pair meets -- both encoders, MLPLocalPre{Fpc,Rpc} and the mrpc boundary head -- depends on one cloud
 * only, so pz_encode_pieces runs it once per piece, and pz_predict_pairs evaluates any list of (i, j) pairs from that
 * state with the pose MLP and the fpc boundary head alone.  Per-piece state, caller-owned, for P pieces:
 * role 0 = the piece as fpc (Encoder, MLPLocalPreFpc), role 1 = the piece as mrpc (Encoder2, MLPLocalPreRpc).
 * Every buffer must be 16-byte aligned (PZ_ERR_ARG otherwise). */
#define PZ_MAX_PIECES 4095      /* pieces per pz_encode_pieces call */
#define PZ_MAX_PAIRS (1 << 20)  /* pairs per pz_predict_pairs call */
typedef struct PzPieceEmbeddings {
  float* f_global; /* [2,P,1024]    f_global of the piece through Encoder (role 0) and Encoder2 (role 1) */
  float* local;    /* [2,P,1024,64] MLPLocalPreFpc(x_feature_E) (role 0), MLPLocalPreRpc(x_feature_E2) (role 1) */
  float* tilemax;  /* [2,P,8,64]    column maxima of each role's local features per 128-point tile; the max over a
                    *               role-1 piece's 8 tiles is the D6 global feature of that piece as mrpc */
  float* de_mrpcb; /* [P,2,1024]    mrpc boundary logits: they depend on the mrpc piece only */
} PzPieceEmbeddings;

/* clouds [P,1024,3]; starts [4,P] in pz_predict5's order (Encoder s1, Encoder s2, Encoder2 s1, Encoder2 s2).
 * Runs pz_predict5's front half on the batch [clouds; clouds] and fills every field of *emb_host.  With the same
 * clouds and starts, the embeddings of piece p are those pz_predict5(fpc = mrpc = clouds) forms for pair p.
 * flags: PZ_FLAG_REUSE_PACKS as in pz_predict5 (PZ_FLAG_NEED is not supported).  Supported: 1 <= P <= PZ_MAX_PIECES
 * (encode larger sets in several calls), precision
 * fp32 / bf16 / split. */
size_t pz_encode_pieces_workspace_bytes(int P);
int pz_encode_pieces(const PzEncoderWeights* enc_host /*[2]*/, const PzHeadWeights* heads_host, const float* clouds,
                     int P, const int64_t* starts, int precision, int flags, const PzPieceEmbeddings* emb_host,
                     void* workspace, size_t workspace_bytes, pz_stream_t stream);

/* pairs [n,2] int64 (i = fpc piece, j = mrpc piece; i == j and repeats allowed; indices must lie in [0,P))
 * -> out6 [n,6], de_fpcb [n,2,1024], de_mrpcb [n,2,1024]: what pz_predict5 returns for the pair (clouds[i], clouds[j])
 * with the starts the pieces were encoded with, computed by the same kernels (pose MLP on [f_global[0,i],
 * f_global[1,j]]; fpc boundary head on local[0,i] with the global feature of piece j; de_mrpcb[j] copied).
 * emb_host must have been filled by pz_encode_pieces with the same weights and precision.  n == 0 is a no-op.
 * de_mrpcb must be 16-byte aligned.  Supported: P >= 1, n <= PZ_MAX_PAIRS (split larger lists).
 * flags: PZ_FLAG_REUSE_PACKS as in pz_predict5. */
size_t pz_predict_pairs_workspace_bytes(int n);
int pz_predict_pairs(const PzHeadWeights* heads_host, const PzPieceEmbeddings* emb_host, int P, const int64_t* pairs,
                     int n, int precision, int flags, float* out6, float* de_fpcb, float* de_mrpcb, void* workspace,
                     size_t workspace_bytes, pz_stream_t stream);

/* se3.exp(x) -- se_math/se3.py:57-80.  twist [B,6] (omega, v) -> g [B,4,4]. */
int pz_se3_exp(const float* twist, int B, float* g, pz_stream_t stream);
/* Its backward: dtwist [B,6] = sum_e dg[b,e] * d g[b,e] / d twist[b,:] over the 12 non-constant entries (rows 0..2)
 * of g; dg [B,4,4].  Same formulas as pz_se3_exp, Taylor branch for |omega| < 0.01 included.  B >= 1. */
int pz_se3_exp_backward(const float* twist, const float* dg, int B, float* dtwist, pz_stream_t stream);

/* ------------------------------------------------- losses / post-forward epilogue */

/* TouchedRegraster.chamfer_loss(a, b) -- model5_b.py:1495-1505 (dataset.py:1135-1145 is the same code):
 * P[b,i,j] = (|x_i|^2 + |y_j|^2) - 2 x_i.y_j in fp32 (the expanded form the reference gets from three bmm's; it
 * can go slightly negative).  x [B,n,3], y [B,m,3] -> min_over_x [B,m] = torch.min(P,1)[0],
 * min_over_y [B,n] = torch.min(P,2)[0]; arg_* (int32, optional) are the minimising indices (first on ties). */
int pz_chamfer(const float* x, const float* y, int B, int n, int m, float* min_over_x, float* min_over_y,
               int32_t* arg_x_or_null, int32_t* arg_y_or_null, pz_stream_t stream);
/* autograd of the above through the arg-mins: grad_x [B,n,3], grad_y [B,m,3] (overwritten). */
int pz_chamfer_grad(const float* x, const float* y, int B, int n, int m, const int32_t* arg_x, const int32_t* arg_y,
                    const float* grad_min_over_x, const float* grad_min_over_y, float* grad_x, float* grad_y,
                    pz_stream_t stream);

/* TouchedRegraster.comp(g, igt) -- model5_b.py:1512-1519: mse(g.igt, I)*16 -> loss [1]. */
int pz_comp(const float* g, const float* igt, int B, float* loss, pz_stream_t stream);
/* Its backward: dg [B,4,4] = dloss[0] * d comp / d g (dloss is a device scalar).  B >= 1. */
int pz_comp_backward(const float* g, const float* igt, int B, const float* dloss, float* dg, pz_stream_t stream);

/* se3.transform(g, a) -- se_math/se3.py:110-120 for points stored [B,n,3]: out = R p + t. */
int pz_se3_transform(const float* g, const float* pts, int B, int n, float* out, pz_stream_t stream);

/* torch.topk(torch.softmax(logits, 1)[:, 1, :], K, 1)[1] -- model5_b.py:1323-1330 (test) / :1085-1092 (train).
 * logits [B,2,N] -> idx [B,K] by descending class-1 probability (ties: lowest index first),
 * prob_or_null [B,K].  Supported: N <= 1024. */
int pz_boundary_topk(const float* logits, int B, int N, int K, int64_t* idx, float* prob_or_null,
                     pz_stream_t stream);

/* torch.topk(values, K, 1) (largest != 0) or torch.topk(-values, K, 1) (largest == 0) for rows of N <= 1024 floats:
 * get_boundary, dataset.py:1359-1362, and the attention top-k of training_step, model5_b.py:939-942.
 * idx [B,K] in selection order (ties: lowest index first), vals_or_null [B,K] the selected values. */
int pz_topk(const float* values, int B, int N, int K, int largest, int64_t* idx, float* vals_or_null,
            pz_stream_t stream);

/* The whole post-forward part of test_step (model5_b.py:1314-1358 with metrics.py:7-10, :54-84) in one
 * launch, one CTA per pair: se3.exp(out6), boundary top-128 of both clouds, gather, alignment of the second
 * boundary by the predicted pose, the boundary chamfer distances, IoU counts and the isotropic pose errors.
 * fpc, src [B,1024,3] (src = rpc in test_step; mrpc for assembly scoring), fpcb/rpcb [B,128,3],
 * fpc_idx/rpc_idx [B,1024] (0/1 floats), igt [B,4,4]; any *_or_null input disables the columns that need it.
 * scores [B,PZ_SCORE_COLS]:
 *   0 isotropic rotation error (deg)   1 isotropic translation error   2 translation mse   3 translation mae
 *   4 |pred & gt| fpc   5 |pred | gt| fpc   6 |pred & gt| mrpc   7 |pred | gt| mrpc   (IoU = sum(4)/sum(5) over the batch)
 *   8 cd_fpc = mean+mean of chamfer_loss(fpcb, de_fpcb)    9 cd_rpc = chamfer_loss(rpcb, aligned de_rpcb)
 *   10 chamfer_loss(de_fpcb, aligned de_mrpcb) -- the pair score used by the assembly driver   11 reserved (0)
 * idx_f/idx_m [B,128] selected indices, bnd_f/bnd_m [B,128,3] the gathered (bnd_m: aligned) boundary points. */
#define PZ_SCORE_COLS 12
int pz_pair_score(const float* out6, const float* de_fpcb, const float* de_mrpcb, const float* fpc,
                  const float* src, const float* fpcb_or_null, const float* rpcb_or_null,
                  const float* fpc_idx_or_null, const float* rpc_idx_or_null, const float* igt_or_null, int B,
                  float* scores, int64_t* idx_f_or_null, int64_t* idx_m_or_null, float* bnd_f_or_null,
                  float* bnd_m_or_null, pz_stream_t stream);

/* ---------------------------------------------------------------- training */
/* Building blocks of the training step (TouchedRegraster.training_step, model5_b.py:912-1155, Adam per
 * :1453-1457).  The reference gets its backward pass from torch autograd; here every op of the graph has an
 * explicit kernel and puzzlenet_b200/training.py sequences them.  fp32 throughout, like the reference (no AMP). */

/* C = epilogue(alpha * op(A) op(B) + beta * C), row-major.  op(A) is M x K: A[m*lda + k], or with transA the
 * stored matrix is K x M: A[k*lda + m]; likewise op(B) is K x N.  batch > 1: independent problems at
 * A + i*strideA, ... (mask and residual use strideC).  Epilogue order: + bias[n], + beta*C, ReLU (relu != 0),
 * zero where mask[m*ldmask + n] <= 0 (the ReLU gate of a backward GEMM), + residual[m*ldres + n].
 * splitk > 1 splits K over CTAs and atomically ADDS alpha*partial into C (pre-zero C; no batching / epilogue):
 * used for weight gradients dW = dY^T X whose K is the row count (up to 2.1 M). */
int pz_sgemm(int transA, int transB, int M, int N, int K, float alpha, const float* A, long long lda,
             const float* B, long long ldb, float beta, float* C, long long ldc, int batch, long long strideA,
             long long strideB, long long strideC, int splitk, const float* bias_or_null, int relu,
             const float* mask_or_null, long long ldmask, const float* residual_or_null, long long ldres,
             pz_stream_t stream);
/* The same product on the tcgen05 tensor cores in TF32 (fp32 in memory, operands rounded to a 10-bit mantissa by
 * the MMA, fp32 accumulate) -- what stock PyTorch 1.10, the version the reference pins, runs nn.Linear with on
 * Ampere-or-newer GPUs.  C[m,n] = sum_k A(m,k) B(n,k); an operand is K-major (A[m*lda + k], B[n*ldb + k]) or, with
 * *_mn_major != 0, MN-major (A[k*lda + m], B[k*ldb + n]).  Epilogue: + bias[n], + C (accumulate), ReLU, mask gate.
 * splitk > 1: K is split over the persistent grid and partial tiles are atomically ADDED into C (pre-zero it).
 * Supported: M % 128 == 0, N % 64 == 0, K % 32 == 0, 16-byte aligned rows. */
int pz_gemm_tf32(int a_mn_major, int b_mn_major, int M, int N, int K, const float* A, long long lda, const float* B,
                 long long ldb, float* C, long long ldc, int splitk, const float* bias_or_null, int relu,
                 const float* mask_or_null, long long ldmask, int accumulate, pz_stream_t stream);
/* batch independent problems (the per-cloud attention products): operand i at A + i*strideA, B + i*strideB, output and
 * mask at + i*strideC; splitk must be 1. */
int pz_gemm_tf32_batched(int a_mn_major, int b_mn_major, int M, int N, int K, const float* A, long long lda,
                         const float* B, long long ldb, float* C, long long ldc, int batch, long long strideA,
                         long long strideB, long long strideC, int splitk, const float* bias_or_null, int relu,
                         const float* mask_or_null, long long ldmask, int accumulate, pz_stream_t stream);
/* Layer 1 of a grouped MLP without the [B,S,K,3+D] tensor (model5_b.py:449-452 with pointnet_util.py:123-130):
 * W1 [xyz_j - c_s ; f_j] + b1 = P_j - Q_s with P [clouds*N, C] per source point and Q [groups, C] per centroid, so
 *   out[r,:] = relu(P[cloud*N + idx[r], :] - Q[r / K, :]),  r = (cloud*S + s)*K + k,  groups = clouds*S,
 * and its backward for a gradient d [groups*K, C] w.r.t. the pre-activation (already ReLU-gated):
 *   dP[cloud*N + idx[r], :] += d[r,:]  (dP is accumulated into),  dQ[g,:] = -sum_k d[g*K + k, :]  (overwritten). */
int pz_gather_sub_relu(const float* P, const float* Q, const int64_t* idx, long long groups, int K, int S, int N, int C,
                       float* out, pz_stream_t stream);
int pz_group_scatter_grad(const float* d, const int64_t* idx, long long groups, int K, int S, int N, int C, float* dP,
                          float* dQ, pz_stream_t stream);
/* softmax(scale * S) over the last dimension of S [rows, L] (model5_b.py:70-72 forward). */
int pz_softmax_forward(const float* S, long long rows, int L, float scale, float* A, pz_stream_t stream);
/* out[n] = beta*out[n] + sum_m x[m*ld + n]  (bias gradients). */
int pz_colsum(const float* x, long long ld, long long M, int N, float beta, float* out, pz_stream_t stream);
/* out[r,c] = a*x[r,c] + b*y[r,c] with row strides (y may be null). */
int pz_axpby(long long rows, int cols, float a, const float* x, long long ldx, float b, const float* y_or_null,
             long long ldy, float* out, long long ldo, pz_stream_t stream);
/* x = act(x + bias[c]) in place, strided 2-D: finishes a split-K forward GEMM (the skinny pose-MLP layers, M = 64). */
int pz_bias_act(long long rows, int cols, float* x, long long ld, const float* bias_or_null, int relu,
                pz_stream_t stream);
/* out = mask > 0 ? dy : 0 (ReLU gate on an incoming gradient), strided 2-D. */
int pz_relu_gate(long long rows, int cols, const float* dy, long long ldy, const float* mask, long long ldm,
                 float* out, long long ldo, pz_stream_t stream);
/* x.repeat(1, reps, 1) of per-cloud rows (model5_b.py:742, :744): dst[(g*reps + r)*ldd + c] = src[g*C + c]; and its
 * backward y[g,c] = sum_k x[(g*K + k)*ld + c]. */
int pz_broadcast_rows(const float* src, long long G, int reps, int C, float* dst, long long ldd, pz_stream_t stream);
int pz_group_sum(const float* x, long long ld, long long G, int K, int C, float* y, pz_stream_t stream);
/* nn.BatchNorm1d(P) applied to x [B,P,C] in TRAIN mode (model5_b.py:424-425, :447-448: the "channel" is the point
 * index, statistics over the B*C values of a point; eps 1e-5, momentum 0.1, unbiased running variance), with the
 * following ReLU fused when relu != 0.  save_mean/save_invstd [P] feed the backward. */
int pz_bn_point_train_forward(const float* x, int B, int P, int C, const float* gamma, const float* beta,
                              float* running_mean_or_null, float* running_var_or_null, float momentum, float eps,
                              int relu, float* y, float* save_mean, float* save_invstd, pz_stream_t stream);
/* accumulate != 0: dgamma / dbeta are added to (a module applied twice per step, predict6). */
int pz_bn_point_train_backward(const float* x, const float* y, const float* dy, int B, int P, int C,
                               const float* gamma, const float* save_mean, const float* save_invstd, int relu,
                               int accumulate, float* dx, float* dgamma, float* dbeta, pz_stream_t stream);
/* torch.max(x, dim=-2) of x [G,K,C] with the arg-max (model5_b.py:454, :461, :474, :741) and its backward;
 * relu_gate != 0 additionally applies the ReLU gate of the layer that produced x (dx is then the gradient of
 * that layer's pre-activation). */
int pz_maxpool_forward(const float* x, long long G, int K, int C, float* y, int32_t* arg, pz_stream_t stream);
int pz_maxpool_backward(const float* dy, const float* y, const int32_t* arg, long long G, int K, int C,
                        int relu_gate, float* dx, pz_stream_t stream);
/* backward of index_points (pointnet_util.py:39-50): dst[(m / per_cloud)*N + idx[m], 0:C] += src[m, c0:c0+C]. */
int pz_scatter_add_rows(const float* src, long long ld, int c0, int C, const int64_t* idx, long long M,
                        long long per_cloud, int N, float* dst, long long ldd, pz_stream_t stream);
/* backward of softmax(S * scale) w.r.t. S (model5_b.py:70-72): dS = scale * A * (dA - rowsum(dA*A)). */
int pz_softmax_backward(const float* A, const float* dA, long long rows, int L, float scale, float* dS,
                        pz_stream_t stream);
/* F.cross_entropy(logits [B,2,N], target [B,N]) (model5_b.py:1063-1064): loss[0] += mean CE (zero it first);
 * dlogits_or_null = grad_scale * d(mean CE)/dlogits.  point_major != 0: logits / dlogits are stored [B,N,2] (the
 * layout the segmentation head produces before the reference's permute, model5_b.py:752). */
int pz_cross_entropy(const float* logits, const float* target, int B, int N, int point_major, float grad_scale,
                     float* loss, float* dlogits_or_null, pz_stream_t stream);
/* d loss / d twist through mat = se3.exp(out6), q = R p + t (model5_b.py:947-949) and, when igt is given,
 * comp_scale * comp(mat, igt) (model5_b.py:963-967):  dout6 = beta*dout6 + J^T(dR, dt), with
 * dR = sum_n dpts_n p_n^T, dt = sum_n dpts_n.  pts/dpts [B,n,3] (both may be null: comp term only). */
int pz_pose_grad(const float* out6, const float* pts_or_null, const float* dpts_or_null, int n,
                 const float* igt_or_null, float comp_scale, int B, float beta, float* dout6, pz_stream_t stream);
/* torch.optim.Adam (model5_b.py:1454; betas, eps as given) on flat buffers; grads are multiplied by grad_scale
 * first (1/world_size after a sum all-reduce). */
int pz_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                 float beta1, float beta2, float eps, int step, float grad_scale, pz_stream_t stream);

/* --------------------------------------------------------------------- EMD */

/* emd_cuda.approxmatch_forward(xyz1, xyz2) -- PyTorchEMD/cuda/emd_kernel.cu:171-193 (kernel :25-158).
 * xyz1 [b,n,3], xyz2 [b,m,3] -> match [b,m,n].  workspace: pz_emd_workspace_bytes(b,n,m). */
size_t pz_emd_workspace_bytes(int b, int n, int m);
int pz_emd_approxmatch(const float* xyz1, const float* xyz2, int b, int n, int m, float* match,
                       void* workspace, size_t workspace_bytes, pz_stream_t stream);
/* emd_cuda.matchcost_forward -- emd_kernel.cu:257-279 (kernel :200-243) -> cost [b]. */
int pz_emd_matchcost(const float* xyz1, const float* xyz2, const float* match, int b, int n, int m,
                     float* cost, pz_stream_t stream);
/* emd_cuda.matchcost_backward -- emd_kernel.cu:373-398 (kernels :286-355) -> grad1 [b,n,3], grad2 [b,m,3]. */
int pz_emd_matchcost_grad(const float* grad_cost, const float* xyz1, const float* xyz2,
                          const float* match, int b, int n, int m, float* grad1, float* grad2,
                          pz_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PUZZLENET_B200_H_ */
