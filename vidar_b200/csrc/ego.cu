// Ego-motion alignment on the device, B200 (sm_100a).
//
//   bev_rotate_kernel      the previous BEV rotated by the ego yaw change about `rotate_center`:
//                          PerceptionTransformer.get_bev_features (bevformer/modules/transformer.py:136-149)
//                          calls torchvision.transforms.functional.rotate(img[C,H,W], angle, center) once per
//                          sample, with its defaults (nearest, expand=False, zero fill) on a permuted copy.
//                          Here the BEV stays channel-last [bs, H*W, C]; one warp per output cell finds the
//                          source cell with torchvision's statements and copies (or zeroes) the C-float row.
//   ego_align_points_kernel  GT points of frame src moved into frame tgt (ViDARHeadV1._get_reference_gt_points,
//                          dense_heads/vidar_head_v1.py:94-148) without the per-frame boolean masks: one thread
//                          per point, `[x y z 1] @ M[b, slot]`; points of frames without a slot become
//                          (NaN, NaN, NaN, -1) in place, so the output keeps the input order.
//
// Both take their per-sample matrices as kernel arguments (host metadata): no H2D copy, no host sync.
// Arithmetic is the reference's fp32 statements with explicit round-to-nearest intrinsics (no FMA
// contraction); no atomics, so two calls are bit-identical.
#include <math.h>

#include "common.cuh"

namespace vidar {
namespace {

constexpr int kRotThreads = 256;             // 8 warps = 8 output cells per block
constexpr int kRotMaxSamples = 32;           // samples per launch (θ travels in the kernel arguments)
constexpr int kAlignThreads = 256;
constexpr int kAlignMaxSamples = 32;
constexpr int kAlignMaxMats = 128;           // (sample, slot) matrices per launch: 8 KB of arguments
constexpr int kAlignMaxFrames = 64;

struct RotArgs {
  const float* src;
  float* dst;
  float theta[kRotMaxSamples][6];            // rescaled θᵀ / [w/2, h/2]: rows (x, y, 1), columns (gx, gy)
  int bs, H, W, C;
};

// torchvision _gen_affine_grid + grid_sample(nearest, zeros, align_corners=False):
//   base (x - w/2 + 0.5, y - h/2 + 0.5, 1) @ rescaled -> (gx, gy) in [-1, 1] units;
//   unnormalise ((g + 1) * size - 1) / 2, round half to even, out of range -> zero.
__global__ void __launch_bounds__(kRotThreads) bev_rotate_kernel(const RotArgs A) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long HW = (long long)A.H * A.W;
  const long long cell = (long long)blockIdx.x * (kRotThreads / 32) + warp;
  if (cell >= (long long)A.bs * HW) return;
  const int b = (int)(cell / HW);
  const int q = (int)(cell - (long long)b * HW);
  const int y = q / A.W, x = q - y * A.W;
  const float* t = A.theta[b];
  // linspace(-w/2 + 0.5, w/2 - 0.5, w) has step 1: exact half-integers
  const float bx = __fadd_rn(__fsub_rn((float)x, 0.5f * (float)A.W), 0.5f);
  const float by = __fadd_rn(__fsub_rn((float)y, 0.5f * (float)A.H), 0.5f);
  const float gx = __fadd_rn(__fadd_rn(__fmul_rn(bx, t[0]), __fmul_rn(by, t[2])), t[4]);
  const float gy = __fadd_rn(__fadd_rn(__fmul_rn(bx, t[1]), __fmul_rn(by, t[3])), t[5]);
  const float ix = rintf(__fdiv_rn(__fsub_rn(__fmul_rn(__fadd_rn(gx, 1.f), (float)A.W), 1.f), 2.f));
  const float iy = rintf(__fdiv_rn(__fsub_rn(__fmul_rn(__fadd_rn(gy, 1.f), (float)A.H), 1.f), 2.f));
  const bool inside = ix >= 0.f && ix <= (float)(A.W - 1) && iy >= 0.f && iy <= (float)(A.H - 1);   // NaN -> outside
  const int C = A.C;
  float* out = A.dst + (size_t)cell * C;
  const float* in = inside ? A.src + ((size_t)b * HW + (size_t)((int)iy * A.W + (int)ix)) * C : nullptr;
  if ((C & 3) == 0) {
    float4* o4 = reinterpret_cast<float4*>(out);
    for (int i = lane; i < (C >> 2); i += 32) o4[i] = inside ? ldg4(in + 4 * i) : make_float4(0.f, 0.f, 0.f, 0.f);
  } else {
    for (int i = lane; i < C; i += 32) out[i] = inside ? __ldg(in + i) : 0.f;
  }
}

struct AlignArgs {
  const float* points;                       // [n, 4] (x, y, z, frame) of this chunk's samples
  float* out;                                // [n, 4]
  float* origins;                            // [chunk, S, 3]
  long long offsets[kAlignMaxSamples + 1];   // chunk-relative point offsets
  int slot_of_frame[kAlignMaxFrames];
  float mats[kAlignMaxMats][16];             // [chunk * S] row-major 4x4, p' = p @ M
  int samples, S, num_frames;
};

__device__ __forceinline__ float row_times_col(float x, float y, float z, const float* M, int j) {
  // torch.matmul([x y z 1], M) column j, k = 0..3 in order, no contraction
  return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(x, M[j]), __fmul_rn(y, M[4 + j])), __fmul_rn(z, M[8 + j])),
                   __fmul_rn(1.f, M[12 + j]));
}

__global__ void __launch_bounds__(kAlignThreads) ego_align_points_kernel(const AlignArgs A) {
  const long long n = A.offsets[A.samples];
  const long long i = (long long)blockIdx.x * kAlignThreads + threadIdx.x;
  if (i < n) {
    int b = 0;
    while (b + 1 < A.samples && A.offsets[b + 1] <= i) ++b;
    const float4 p = *reinterpret_cast<const float4*>(A.points + 4 * i);
    int slot = -1;
    if (p.w >= 0.f && p.w < (float)A.num_frames && p.w == truncf(p.w)) slot = A.slot_of_frame[(int)p.w];
    float4 r = make_float4(NAN, NAN, NAN, -1.f);
    if (slot >= 0) {
      const float* M = A.mats[b * A.S + slot];
      r = make_float4(row_times_col(p.x, p.y, p.z, M, 0), row_times_col(p.x, p.y, p.z, M, 1),
                      row_times_col(p.x, p.y, p.z, M, 2), (float)slot);
    }
    *reinterpret_cast<float4*>(A.out + 4 * i) = r;
  } else if (i < n + (long long)A.samples * A.S) {
    const int m = (int)(i - n);                                   // (b, s) = the sensor origin [0 0 0 1] @ M
    const float* M = A.mats[m];
    for (int j = 0; j < 3; ++j) A.origins[(size_t)m * 3 + j] = row_times_col(0.f, 0.f, 0.f, M, j);
  }
}

}  // namespace
}  // namespace vidar

using namespace vidar;

extern "C" int vidar_bev_rotate_forward(const float* src, const float* theta_host, float* dst, int bs, int H, int W,
                                        int C, void* stream) {
  VIDAR_REQUIRE(src && theta_host && dst, "bev_rotate_forward: null pointer argument");
  VIDAR_REQUIRE(bs > 0 && H > 0 && W > 0 && C > 0, "bev_rotate_forward: bad sizes bs=%d H=%d W=%d C=%d", bs, H, W, C);
  VIDAR_REQUIRE(src != dst, "bev_rotate_forward: src and dst must not alias");
  VIDAR_REQUIRE((C & 3) != 0 || ((uintptr_t)src % 16 == 0 && (uintptr_t)dst % 16 == 0),
                "bev_rotate_forward: src and dst must be 16-byte aligned when C %% 4 == 0");
  const long long HW = (long long)H * W;
  for (int b0 = 0; b0 < bs; b0 += kRotMaxSamples) {
    RotArgs A;
    A.bs = bs - b0 < kRotMaxSamples ? bs - b0 : kRotMaxSamples;
    A.H = H; A.W = W; A.C = C;
    A.src = src + (size_t)b0 * HW * C;
    A.dst = dst + (size_t)b0 * HW * C;
    for (int b = 0; b < A.bs; ++b)
      for (int k = 0; k < 6; ++k) A.theta[b][k] = theta_host[(size_t)(b0 + b) * 6 + k];
    const long long cells = (long long)A.bs * HW;
    const long long blocks = (cells + kRotThreads / 32 - 1) / (kRotThreads / 32);
    VIDAR_REQUIRE(blocks <= 2147483647LL, "bev_rotate_forward: grid too large");
    bev_rotate_kernel<<<(unsigned)blocks, kRotThreads, 0, (cudaStream_t)stream>>>(A);
    const int rc = check_launch("bev_rotate_forward");
    if (rc != VIDAR_OK) return rc;
  }
  return VIDAR_OK;
}

extern "C" int vidar_ego_align_points(const float* points, const int64_t* offsets_host,
                                      const int32_t* slot_of_frame_host, int num_frames,
                                      const float* src_to_tgt_host, float* out_points, float* origins, int bs, int S,
                                      void* stream) {
  VIDAR_REQUIRE(offsets_host && slot_of_frame_host && src_to_tgt_host && origins,
                "ego_align_points: null pointer argument");
  VIDAR_REQUIRE(bs > 0 && S > 0 && S <= kAlignMaxMats, "ego_align_points: bad sizes bs=%d S=%d (S <= %d)", bs, S,
                kAlignMaxMats);
  VIDAR_REQUIRE(num_frames > 0 && num_frames <= kAlignMaxFrames, "ego_align_points: num_frames=%d not in [1, %d]",
                num_frames, kAlignMaxFrames);
  VIDAR_REQUIRE(offsets_host[0] == 0, "ego_align_points: offsets must start at 0");
  for (int b = 0; b < bs; ++b)
    VIDAR_REQUIRE(offsets_host[b + 1] >= offsets_host[b], "ego_align_points: offsets must not decrease (sample %d)", b);
  VIDAR_REQUIRE(offsets_host[bs] == 0 || (points && out_points), "ego_align_points: null pointer argument");
  for (int f = 0; f < num_frames; ++f)
    VIDAR_REQUIRE(slot_of_frame_host[f] >= -1 && slot_of_frame_host[f] < S,
                  "ego_align_points: slot_of_frame[%d] = %d not in [-1, S)", f, slot_of_frame_host[f]);
  const int per_launch = kAlignMaxMats / S < kAlignMaxSamples ? kAlignMaxMats / S : kAlignMaxSamples;
  for (int b0 = 0; b0 < bs; b0 += per_launch) {
    AlignArgs A;
    A.samples = bs - b0 < per_launch ? bs - b0 : per_launch;
    A.S = S; A.num_frames = num_frames;
    const long long base = offsets_host[b0];
    for (int b = 0; b <= A.samples; ++b) A.offsets[b] = offsets_host[b0 + b] - base;
    for (int f = 0; f < num_frames; ++f) A.slot_of_frame[f] = slot_of_frame_host[f];
    for (int m = 0; m < A.samples * S; ++m)
      for (int k = 0; k < 16; ++k) A.mats[m][k] = src_to_tgt_host[((size_t)b0 * S + m) * 16 + k];
    A.points = points ? points + 4 * base : nullptr;
    A.out = out_points ? out_points + 4 * base : nullptr;
    A.origins = origins + (size_t)b0 * S * 3;
    const long long work = A.offsets[A.samples] + (long long)A.samples * S;
    const long long blocks = (work + kAlignThreads - 1) / kAlignThreads;
    VIDAR_REQUIRE(blocks <= 2147483647LL, "ego_align_points: grid too large");
    ego_align_points_kernel<<<(unsigned)blocks, kAlignThreads, 0, (cudaStream_t)stream>>>(A);
    const int rc = check_launch("ego_align_points");
    if (rc != VIDAR_OK) return rc;
  }
  return VIDAR_OK;
}
