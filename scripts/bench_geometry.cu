// Harness of scripts/bench_geometry.py: the encoder's geometry as one launch (geometry_c2_kernel with W kNN workers,
// W = 0 is the FPS chains alone) and as the six launches it replaces.  Compiled on its own with geometry.cu included,
// so it can instantiate worker counts the library does not build.
#include "../puzzlenet_b200/csrc/geometry.cu"

namespace pz {
char* error_buffer() {
  static char buf[512];
  return buf;
}
int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(error_buffer(), 512, fmt, ap);
  va_end(ap);
  return code;
}
void count_launch() {}
bool pdl_for_stream(cudaStream_t) { return false; }
}  // namespace pz

using namespace pz;

extern "C" const char* geo_last_error() { return error_buffer(); }

// the buffers of one forward's geometry (C clouds, the first B use weight set 0); w1 [128, ldw1], w2 [256, ldw2] per set
static EncoderGeometry geo_args(const float* xyz, const int64_t* s1, const int64_t* s2, int B, int64_t* fps1, int64_t* knn1,
                                int64_t* fps2, int64_t* knn2, float* nx1, float* nx2, int* knn1r, int* knn2r, float* Q1, float* Q2,
                                const float* w1a, const float* w1b, int ldw1, const float* w2a, const float* w2b, int ldw2) {
  EncoderGeometry g;
  g.xyz = xyz; g.start1 = s1; g.start2 = s2;
  g.fps1 = fps1; g.knn1 = knn1; g.fps2 = fps2; g.knn2 = knn2;
  g.nx1 = nx1; g.nx2 = nx2; g.knn1r = knn1r; g.knn2r = knn2r; g.Q1 = Q1; g.Q2 = Q2;
  g.w1[0] = w1a; g.w1[1] = w1b; g.ldw1 = ldw1; g.w2[0] = w2a; g.w2[1] = w2b; g.ldw2 = ldw2;
  g.clouds_per_set = B;
  return g;
}

extern "C" int geo_fused(int W, const float* xyz, const int64_t* s1, const int64_t* s2, int C, int B, int64_t* fps1,
                         int64_t* knn1, int64_t* fps2, int64_t* knn2, float* nx1, float* nx2, int* knn1r, int* knn2r, float* Q1,
                         float* Q2, const float* w1a, const float* w1b, int ldw1, const float* w2a, const float* w2b, int ldw2,
                         void* stream) {
  const EncoderGeometry g = geo_args(xyz, s1, s2, B, fps1, knn1, fps2, knn2, nx1, nx2, knn1r, knn2r, Q1, Q2, w1a, w1b, ldw1,
                                     w2a, w2b, ldw2);
  const cudaStream_t st = (cudaStream_t)stream;
  switch (W) {
    case 0: return launch_encoder_geometry_w<0>(g, C, st);
    case 8: return launch_encoder_geometry_w<8>(g, C, st);
    case 12: return launch_encoder_geometry_w<12>(g, C, st);
    case 16: return launch_encoder_geometry_w<16>(g, C, st);
    default: return fail(PZ_ERR_ARG, "geo_fused: W=%d not built", W);
  }
}

extern "C" int geo_separate(const float* xyz, const int64_t* s1, const int64_t* s2, int C, int B, int64_t* fps1, int64_t* knn1,
                            int64_t* fps2, int64_t* knn2, float* nx1, float* nx2, int* knn1r, int* knn2r, float* Q1, float* Q2,
                            const float* w1a, const float* w1b, int ldw1, const float* w2a, const float* w2b, int ldw2,
                            void* stream) {
  const cudaStream_t st = (cudaStream_t)stream;
  PZ_TRY(launch_fps(xyz, C, 1024, s1, 512, fps1, nullptr, nx1, st));
  PZ_TRY(launch_knn(nx1, xyz, C, 512, 1024, 32, knn1, knn1r, nullptr, st));
  if (Q1) PZ_TRY(launch_centre_proj_f32(nx1, w1a, w1b, ldw1, B * 512, C * 512, 128, Q1, st));
  PZ_TRY(launch_fps(nx1, C, 512, s2, 256, fps2, nullptr, nx2, st));
  PZ_TRY(launch_knn(nx2, nx1, C, 256, 512, 32, knn2, knn2r, nullptr, st));
  if (Q2) PZ_TRY(launch_centre_proj_f32(nx2, w2a, w2b, ldw2, B * 256, C * 256, 256, Q2, st));
  return 0;
}
