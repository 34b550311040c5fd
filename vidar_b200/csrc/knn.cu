// Nearest-neighbour (K = 1) search and its backward for the Chamfer distance, B200 (sm_100a).
//
// Reference: third_lib/chamfer_dist/chamferdist/chamferdist/knn.cu:21-260 (brute-force KNN,
// 256 blocks x 256 threads, every thread scans all of P2 from global memory), knn_cpu.cpp:7-106,
// used with K = 1 by ChamferDistance (chamfer.py:20-133) for ViDAR's evaluation metric
// (bevformer/utils/e2e_predictor_utils.py:163-183) -- SURVEY.md 8(f) item 2.
// dist = sum_d (p1 - p2)^2 accumulated in d order like the CPU reference; ties keep the
// smallest index (the CPU loop keeps the first strictly-smaller candidate).
//
// Mapping: a thread owns one p1 point; p2 streams through shared memory in 1024-point tiles
// (12 KB, read once per block instead of once per thread), and P2 is additionally split over
// blockIdx.y so 30k x 30k points fill all 148 SMs; partial results merge with one 64-bit
// atomicMin on (distance bits << 32 | index) -- non-negative floats order like unsigned ints.
#include "common.cuh"

namespace vidar {
namespace {

constexpr int kNnThreads = 256;
constexpr int kNnTile = 1024;

template <int D>
__global__ void __launch_bounds__(kNnThreads)
nn_forward_kernel(const float* __restrict__ p1, const float* __restrict__ p2,
                  const int64_t* __restrict__ len1, const int64_t* __restrict__ len2,
                  unsigned long long* __restrict__ best, int N, int P1, int P2, int splits) {
  __shared__ float tile[kNnTile * D];
  const int n = blockIdx.z;
  const int i = blockIdx.x * kNnThreads + threadIdx.x;
  const int L1 = len1 ? (int)len1[n] : P1;
  const int L2 = len2 ? (int)len2[n] : P2;
  const int chunk = (L2 + splits - 1) / splits;
  const int j0 = blockIdx.y * chunk, j1 = min(L2, j0 + chunk);
  // nothing to do: no P2 points in this split, or (launched over an upper bound P1) no live p1 point
  if (j0 >= j1 || (int)(blockIdx.x * kNnThreads) >= L1) return;
  float a[D];
  const bool live = i < L1;
#pragma unroll
  for (int d = 0; d < D; ++d) a[d] = live ? p1[((size_t)n * P1 + i) * D + d] : 0.f;
  float bd = INFINITY;
  int bi = 0;
  for (int t0 = j0; t0 < j1; t0 += kNnTile) {
    const int cnt = min(kNnTile, j1 - t0);
    __syncthreads();
    for (int e = threadIdx.x; e < cnt * D; e += kNnThreads) tile[e] = p2[((size_t)n * P2 + t0) * D + e];
    __syncthreads();
    if (live) {
      for (int j = 0; j < cnt; ++j) {
        float dist = 0.f;
#pragma unroll
        for (int d = 0; d < D; ++d) {
          const float diff = a[d] - tile[j * D + d];
          dist = __fadd_rn(dist, __fmul_rn(diff, diff));     // `dist += diff * diff`, no contraction
        }
        if (dist < bd) { bd = dist; bi = t0 + j; }
      }
    }
  }
  if (live) {
    const unsigned long long key = ((unsigned long long)__float_as_uint(bd) << 32) | (unsigned)bi;
    atomicMin(best + (size_t)n * P1 + i, key);
  }
}

__global__ void nn_unpack_kernel(const unsigned long long* __restrict__ best, const int64_t* __restrict__ len1,
                                 const int64_t* __restrict__ len2, float* __restrict__ dists,
                                 int64_t* __restrict__ idx, int N, int P1, int P2) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)N * P1) return;
  const int n = (int)(t / P1), i = (int)(t % P1);
  const int L1 = len1 ? (int)len1[n] : P1;
  const int L2 = len2 ? (int)len2[n] : P2;
  const unsigned long long key = best[t];
  const bool ok = i < L1 && L2 > 0 && key != ~0ull;
  dists[t] = ok ? __uint_as_float((unsigned)(key >> 32)) : 0.f;     // zero padding like the reference
  idx[t] = ok ? (int64_t)(unsigned)(key & 0xffffffffu) : 0;
}

template <int D>
__global__ void nn_backward_kernel(const float* __restrict__ p1, const float* __restrict__ p2,
                                   const int64_t* __restrict__ len1, const int64_t* __restrict__ len2,
                                   const int64_t* __restrict__ idx, const float* __restrict__ grad_dists,
                                   float* __restrict__ grad_p1, float* __restrict__ grad_p2, int N, int P1,
                                   int P2) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)N * P1) return;
  const int n = (int)(t / P1), i = (int)(t % P1);
  const int L1 = len1 ? (int)len1[n] : P1;
  const int L2 = len2 ? (int)len2[n] : P2;
  if (i >= L1 || L2 < 1) return;
  const int64_t j = idx[t];
  const float g = grad_dists[t];
#pragma unroll
  for (int d = 0; d < D; ++d) {
    const float diff = 2.0f * g * (p1[t * D + d] - p2[((size_t)n * P2 + j) * D + d]);
    grad_p1[t * D + d] = diff;                                 // caller-zeroed, one writer
    red_add_f32(grad_p2 + ((size_t)n * P2 + j) * D + d, -diff);
  }
}

}  // namespace
}  // namespace vidar

using namespace vidar;

extern "C" int vidar_nn_forward(const float* p1, const float* p2, const int64_t* lengths1,
                                const int64_t* lengths2, float* dists, int64_t* idx,
                                unsigned long long* scratch, int N, int P1, int P2, int D, void* stream) {
  VIDAR_REQUIRE(p1 && p2 && dists && idx && scratch, "knn_points: null pointer argument");
  VIDAR_REQUIRE(N > 0 && P1 > 0 && P2 > 0, "knn_points: bad sizes N=%d P1=%d P2=%d", N, P1, P2);
  VIDAR_REQUIRE(D == 2 || D == 3 || D == 4, "knn_points: point dimension %d unsupported (2, 3 or 4)", D);
  VIDAR_REQUIRE(N <= 65535, "knn_points: batch too large");
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(scratch, 0xff, sizeof(unsigned long long) * (size_t)N * P1, st);
  if (e != cudaSuccess) return set_error(VIDAR_E_CUDA, "knn_points: memset: %s", cudaGetErrorString(e));
  const int bx = (P1 + kNnThreads - 1) / kNnThreads;
  // enough (block x split) pairs for ~4 waves of 148 SMs, at least one tile per split
  int splits = (4 * kNumSMs + bx * N - 1) / (bx * N);
  const int max_splits = (P2 + kNnTile - 1) / kNnTile;
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  const dim3 grid(bx, splits, N);
  if (D == 3) nn_forward_kernel<3><<<grid, kNnThreads, 0, st>>>(p1, p2, lengths1, lengths2, scratch, N, P1, P2, splits);
  else if (D == 2) nn_forward_kernel<2><<<grid, kNnThreads, 0, st>>>(p1, p2, lengths1, lengths2, scratch, N, P1, P2, splits);
  else nn_forward_kernel<4><<<grid, kNnThreads, 0, st>>>(p1, p2, lengths1, lengths2, scratch, N, P1, P2, splits);
  int rc = check_launch("knn_points");
  if (rc) return rc;
  const long long total = (long long)N * P1;
  nn_unpack_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(scratch, lengths1, lengths2, dists, idx, N, P1, P2);
  return check_launch("knn_points(unpack)");
}

extern "C" int vidar_nn_backward(const float* p1, const float* p2, const int64_t* lengths1,
                                 const int64_t* lengths2, const int64_t* idx, const float* grad_dists,
                                 float* grad_p1, float* grad_p2, int N, int P1, int P2, int D, void* stream) {
  VIDAR_REQUIRE(p1 && p2 && idx && grad_dists && grad_p1 && grad_p2, "knn_points_backward: null pointer argument");
  VIDAR_REQUIRE(N > 0 && P1 > 0 && P2 > 0, "knn_points_backward: bad sizes");
  VIDAR_REQUIRE(D == 2 || D == 3 || D == 4, "knn_points_backward: point dimension %d unsupported", D);
  const long long total = (long long)N * P1;
  const unsigned nb = (unsigned)((total + 255) / 256);
  cudaStream_t st = (cudaStream_t)stream;
  if (D == 3) nn_backward_kernel<3><<<nb, 256, 0, st>>>(p1, p2, lengths1, lengths2, idx, grad_dists, grad_p1, grad_p2, N, P1, P2);
  else if (D == 2) nn_backward_kernel<2><<<nb, 256, 0, st>>>(p1, p2, lengths1, lengths2, idx, grad_dists, grad_p1, grad_p2, N, P1, P2);
  else nn_backward_kernel<4><<<nb, 256, 0, st>>>(p1, p2, lengths1, lengths2, idx, grad_dists, grad_p1, grad_p2, N, P1, P2);
  return check_launch("knn_points_backward");
}
