// Point-cloud forecasting metrics (Chamfer-inner, ray L1 / AbsRel) on the device, B200 (sm_100a).
//
// Reference: ViDAR.forward_test (projects/mmdet3d_plugin/bevformer/detectors/vidar.py:389-502) scores
// every (sample, frame) on the host: boolean-mask compaction of the decoded clouds
// (dense_heads/vidar_head_base.py:344-389, utils/e2e_predictor_utils.py:146-184), `.cpu().numpy()`
// copies and a numpy ray clamp with Python loops over rays (utils/eval_utils.py `clamp`, `_clamp`,
// `spherical_projection`, `compute_ray_errors`).  Here one segment = one (batch element, frame):
//
//   eval_gather_kernel      one block per segment: selects the frame's rays, forms the predicted and
//                           GT points with get_rendered_pcds' fp32 statements and compacts four
//                           stably ordered lists with a ballot + block scan (like sca_compact_kernel):
//                           (0) pred inside pc_range, (1) GT inside pc_range,
//                           (2) pred spherical (atan2(x,y), atan2(z,y), 1) with d_hat > 1e-2, + d_hat,
//                           (3) GT spherical with d > 1e-2, + the GT point.
//   (vidar_nn_forward)      nearest neighbours between the lists, lengths read from device memory.
//   eval_ray_errors_kernel  one block per segment: per GT ray of list (3) the interpolated point,
//                           both clamped to the eval box with the exact semantics of eval_utils'
//                           clamp / _clamp, Σ eucl and Σ eucl / d_clamped; plus the two Chamfer sums.
//                           Sums run in fp64 over a fixed thread assignment and a fixed reduction tree
//                           (no atomics): two calls are bit-identical.
//
// Precision: every per-ray statement is the reference's fp32 numpy / torch statement with explicit
// round-to-nearest intrinsics (no FMA contraction).  Under numpy >= 2 (NEP 50) the plane distances,
// `isclose` and the inside_volume bounds of the clamp are float32 as well: python-float operands take
// the array's dtype.  atan2 is evaluated in fp64 and rounded once (correctly rounded in fp32).
#include <math.h>

#include "common.cuh"

namespace vidar {
namespace {

constexpr int kGatherThreads = 1024;
constexpr int kErrThreads = 256;

// eval_utils.PC_RANGE and inside_volume's 0.02 slack, rounded to fp32 as numpy compares them
__constant__ float kBoxLo[3] = {-70.0f, -70.0f, -4.5f};
__constant__ float kBoxHi[3] = {70.0f, 70.0f, 4.5f};
__constant__ float kSlackLo[3] = {(float)(-70.0 - 0.02), (float)(-70.0 - 0.02), (float)(-4.5 - 0.02)};
__constant__ float kSlackHi[3] = {(float)(70.0 + 0.02), (float)(70.0 + 0.02), (float)(4.5 + 0.02)};

struct F3 {
  float v[3];
};

__device__ __forceinline__ float norm3(float x, float y, float z) {
  // sqrt(x*x + y*y + z*z) / sqrt((v ** 2).sum(1)): left to right, no contraction
  return __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z)));
}

__device__ __forceinline__ float atan2_rn(float y, float x) { return (float)atan2((double)y, (double)x); }

__device__ __forceinline__ bool inside_range(const float* r, float x, float y, float z) {
  return r[0] <= x && x <= r[3] && r[1] <= y && y <= r[4] && r[2] <= z && z <= r[5];
}

// eval_utils.inside_volume
__device__ __forceinline__ bool inside_volume(const F3& p) {
  return kSlackLo[0] <= p.v[0] && p.v[0] <= kSlackHi[0] && kSlackLo[1] <= p.v[1] && p.v[1] <= kSlackHi[1] &&
         kSlackLo[2] <= p.v[2] && p.v[2] <= kSlackHi[2];
}

// Distances from q to the six box planes along sign * d, `np.where(np.isclose(d, 0), MAX_VALUE, ...)`,
// sorted ascending.  The reference visits the planes in argsort order; what it does at a plane depends on
// the distance value only, so the order among equal values does not matter.
__device__ __forceinline__ void sorted_plane_distances(const F3& q, const float* d, float sign, float* t) {
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const bool close0 = fabsf(d[a]) <= 1e-8f || d[a] == 0.f;
    const float den = sign > 0.f ? d[a] : -d[a];
    t[2 * a] = close0 ? 1e8f : __fdiv_rn(__fsub_rn(kBoxLo[a], q.v[a]), den);
    t[2 * a + 1] = close0 ? 1e8f : __fdiv_rn(__fsub_rn(kBoxHi[a], q.v[a]), den);
  }
#pragma unroll
  for (int i = 1; i < 6; ++i) {
#pragma unroll
    for (int j = i; j > 0; --j) {
      const float lo = fminf(t[j - 1], t[j]), hi = fmaxf(t[j - 1], t[j]);
      t[j - 1] = lo;
      t[j] = hi;
    }
  }
}

// eval_utils.clamp for one point of a cloud sharing `o` (origin_inside = inside_volume(origin)).
// -> clamped origin `no`, clamped point `p` (in place), invalid (all-inf / all-NaN); `err` |= 1 for a
// degenerate ray (the reference raises RuntimeError), |= 2 when `assert(touches_volume)` would fail.
__device__ void clamp_point(const F3& o, bool origin_inside, F3& p, F3& no, bool& invalid, int& err) {
  no = o;
  const bool inner = kBoxLo[0] <= p.v[0] && p.v[0] <= kBoxHi[0] && kBoxLo[1] <= p.v[1] && p.v[1] <= kBoxHi[1] &&
                     kBoxLo[2] <= p.v[2] && p.v[2] <= kBoxHi[2];
  if (!inner) {                                                        // _clamp
    float e[3], d[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) e[a] = __fsub_rn(p.v[a], o.v[a]);
    if (e[0] == 0.f && e[1] == 0.f && e[2] == 0.f) err |= 1;
    const float l = norm3(e[0], e[1], e[2]);
#pragma unroll
    for (int a = 0; a < 3; ++a) d[a] = __fdiv_rn(e[a], l);
    bool hit = origin_inside;
    float t[6];
    if (!origin_inside) {                                              // enter the box from outside
      sorted_plane_distances(o, d, 1.f, t);
      for (int k = 0; k < 6; ++k) {
        if (__fadd_rn(t[k], 1e-4f) >= 0.f) {
          F3 x;
#pragma unroll
          for (int a = 0; a < 3; ++a) x.v[a] = __fadd_rn(o.v[a], __fmul_rn(t[k], d[a]));
          if (inside_volume(x)) {
            hit = true;
            no = x;
            if (t[k] > l) p = x;
            break;
          }
        }
      }
    }
    // distances along the reversed ray from the (possibly moved) end point, with the original direction
    sorted_plane_distances(p, d, -1.f, t);
    if (!hit) {
#pragma unroll
      for (int a = 0; a < 3; ++a) no.v[a] = p.v[a] = INFINITY;
    } else if (!inside_volume(p)) {
      bool touches = false;
      for (int k = 0; k < 6; ++k) {
        if (__fadd_rn(t[k], 1e-4f) >= 0.f) {
          F3 x;
#pragma unroll
          for (int a = 0; a < 3; ++a) x.v[a] = __fadd_rn(p.v[a], __fmul_rn(t[k], -d[a]));
          if (inside_volume(x)) {
            p = x;
            touches = true;
            break;
          }
        }
      }
      if (!touches) err |= 2;
    }
  }
  invalid = (isinf(p.v[0]) && isinf(p.v[1]) && isinf(p.v[2])) || (isnan(p.v[0]) && isnan(p.v[1]) && isnan(p.v[2]));
}

struct GatherArgs {
  const float *origin, *points, *tindex, *gt_dist, *pred_dist;
  float range[6];
  int within, M, F;
  float *pred_in, *gt_in, *pred_sph, *pred_dhat, *gt_sph, *gt_pts;
  int64_t* counts;   // [4, N]
};

__global__ void __launch_bounds__(kGatherThreads) eval_gather_kernel(GatherArgs A) {
  const int s = blockIdx.x, N = gridDim.x;
  const int b = s / A.F, t = s % A.F;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  __shared__ int wt[4][32];
  __shared__ int woff[4][32];
  __shared__ int tot[4];
  const F3 o = {{A.origin[(size_t)s * 3], A.origin[(size_t)s * 3 + 1], A.origin[(size_t)s * 3 + 2]}};
  const float tf = (float)t;
  const size_t seg = (size_t)s * A.M;
  int base[4] = {0, 0, 0, 0};
  for (int i0 = 0; i0 < A.M; i0 += kGatherThreads) {
    const int i = i0 + tid;
    bool f[4] = {false, false, false, false};
    F3 pr, gt;
    float dh = 0.f, az_p = 0.f, el_p = 0.f, az_g = 0.f, el_g = 0.f;
    if (i < A.M) {
      const size_t r = (size_t)b * A.M + i;
      const float px = A.points[r * 3], py = A.points[r * 3 + 1], pz = A.points[r * 3 + 2];
      bool sel = A.tindex[r] == tf;
      if (A.gt_dist) sel = sel && A.gt_dist[r] > 0.f;
      if (A.within) sel = sel && inside_range(A.range, px, py, pz);
      if (sel) {
        if (A.gt_dist) {       // get_rendered_pcds: origin + r / |r| * dist
          const float rx = __fsub_rn(px, o.v[0]), ry = __fsub_rn(py, o.v[1]), rz = __fsub_rn(pz, o.v[2]);
          const float n = norm3(rx, ry, rz);
          const float u[3] = {__fdiv_rn(rx, n), __fdiv_rn(ry, n), __fdiv_rn(rz, n)};
          const float dp = A.pred_dist[r], dg = A.gt_dist[r];
#pragma unroll
          for (int a = 0; a < 3; ++a) {
            pr.v[a] = __fadd_rn(o.v[a], __fmul_rn(u[a], dp));
            gt.v[a] = __fadd_rn(o.v[a], __fmul_rn(u[a], dg));
          }
        } else {               // the points are the cloud itself
          pr.v[0] = gt.v[0] = px;
          pr.v[1] = gt.v[1] = py;
          pr.v[2] = gt.v[2] = pz;
        }
        f[0] = inside_range(A.range, pr.v[0], pr.v[1], pr.v[2]);
        f[1] = inside_range(A.range, gt.v[0], gt.v[1], gt.v[2]);
        // spherical_projection(pcd - origin)
        const float qx = __fsub_rn(pr.v[0], o.v[0]), qy = __fsub_rn(pr.v[1], o.v[1]), qz = __fsub_rn(pr.v[2], o.v[2]);
        dh = norm3(qx, qy, qz);
        f[2] = dh > 1e-2f;
        az_p = atan2_rn(qx, qy);
        el_p = atan2_rn(qz, qy);
        const float vx = __fsub_rn(gt.v[0], o.v[0]), vy = __fsub_rn(gt.v[1], o.v[1]), vz = __fsub_rn(gt.v[2], o.v[2]);
        f[3] = norm3(vx, vy, vz) > 1e-2f;
        az_g = atan2_rn(vx, vy);
        el_g = atan2_rn(vz, vy);
      }
    }
    unsigned bal[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) bal[k] = __ballot_sync(0xffffffffu, f[k]);
    if (lane == 0) {
#pragma unroll
      for (int k = 0; k < 4; ++k) wt[k][warp] = __popc(bal[k]);
    }
    __syncthreads();
    if (warp < 4) {            // warp k: exclusive scan of list k's 32 warp totals
      const int v = wt[warp][lane];
      int inc = v;
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const int nb = __shfl_up_sync(0xffffffffu, inc, off);
        if (lane >= off) inc += nb;
      }
      woff[warp][lane] = inc - v;
      if (lane == 31) tot[warp] = inc;
    }
    __syncthreads();
    const unsigned lt = (1u << lane) - 1u;
    int pos[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) pos[k] = base[k] + woff[k][warp] + __popc(bal[k] & lt);
    if (f[0]) {
      float* q = A.pred_in + (seg + pos[0]) * 3;
      q[0] = pr.v[0]; q[1] = pr.v[1]; q[2] = pr.v[2];
    }
    if (f[1]) {
      float* q = A.gt_in + (seg + pos[1]) * 3;
      q[0] = gt.v[0]; q[1] = gt.v[1]; q[2] = gt.v[2];
    }
    if (f[2]) {
      float* q = A.pred_sph + (seg + pos[2]) * 3;
      q[0] = az_p; q[1] = el_p; q[2] = 1.f;
      A.pred_dhat[seg + pos[2]] = dh;
    }
    if (f[3]) {
      float* q = A.gt_sph + (seg + pos[3]) * 3;
      q[0] = az_g; q[1] = el_g; q[2] = 1.f;
      float* g = A.gt_pts + (seg + pos[3]) * 3;
      g[0] = gt.v[0]; g[1] = gt.v[1]; g[2] = gt.v[2];
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) base[k] += tot[k];
    __syncthreads();           // wt / woff / tot are rewritten by the next chunk
  }
  if (tid < 4) A.counts[(size_t)tid * N + s] = base[tid];
}

// fixed-order block sum of three fp64 values and an int OR; result valid in thread 0
__device__ __forceinline__ void block_reduce(double (&v)[3], int& err) {
  __shared__ double sh[3][kErrThreads / 32];
  __shared__ int she[kErrThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
#pragma unroll
    for (int k = 0; k < 3; ++k) v[k] += __shfl_down_sync(0xffffffffu, v[k], off);
    err |= __shfl_down_sync(0xffffffffu, err, off);
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < 3; ++k) sh[k][warp] = v[k];
    she[warp] = err;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 0; k < 3; ++k) {
      double a = 0.0;
      for (int w = 0; w < kErrThreads / 32; ++w) a += sh[k][w];
      v[k] = a;
    }
    int e = 0;
    for (int w = 0; w < kErrThreads / 32; ++w) e |= she[w];
    err = e;
  }
}

struct ErrArgs {
  const float *origin, *pred_dhat, *gt_pts, *cham_fwd, *cham_bwd;
  const int64_t *nn_idx, *counts;
  double* out;
  int Mp, Mg;
};

__global__ void __launch_bounds__(kErrThreads) eval_ray_errors_kernel(ErrArgs A) {
  const int s = blockIdx.x, N = gridDim.x;
  const int n_pin = (int)A.counts[s], n_gin = (int)A.counts[N + s];
  const int n_psph = (int)A.counts[2 * N + s], n_gsph = (int)A.counts[3 * N + s];
  const F3 o = {{A.origin[(size_t)s * 3], A.origin[(size_t)s * 3 + 1], A.origin[(size_t)s * 3 + 2]}};
  const bool origin_inside = inside_volume(o);
  double acc[3] = {0.0, 0.0, 0.0};   // Σ eucl, Σ eucl / d_clamped, unused
  int err = 0;
  if (n_psph > 0) {
    for (int j = threadIdx.x; j < n_gsph; j += kErrThreads) {
      const size_t r = (size_t)s * A.Mg + j;
      F3 g = {{A.gt_pts[r * 3], A.gt_pts[r * 3 + 1], A.gt_pts[r * 3 + 2]}};
      const float dhat = A.pred_dhat[(size_t)s * A.Mp + A.nn_idx[r]];
      const float vx = __fsub_rn(g.v[0], o.v[0]), vy = __fsub_rn(g.v[1], o.v[1]), vz = __fsub_rn(g.v[2], o.v[2]);
      const float n = norm3(vx, vy, vz);
      const float u[3] = {__fdiv_rn(vx, n), __fdiv_rn(vy, n), __fdiv_rn(vz, n)};
      F3 ip;
#pragma unroll
      for (int a = 0; a < 3; ++a) ip.v[a] = __fadd_rn(o.v[a], __fmul_rn(dhat, u[a]));
      F3 go, io;
      bool inv, inv_i;
      clamp_point(o, origin_inside, g, go, inv, err);
      clamp_point(o, origin_inside, ip, io, inv_i, err);
      if (inv) continue;
      const float dc = norm3(__fsub_rn(g.v[0], go.v[0]), __fsub_rn(g.v[1], go.v[1]), __fsub_rn(g.v[2], go.v[2]));
      if (!(dc > 0.01f)) continue;
      const float e = norm3(__fsub_rn(g.v[0], ip.v[0]), __fsub_rn(g.v[1], ip.v[1]), __fsub_rn(g.v[2], ip.v[2]));
      acc[0] += (double)e;
      acc[1] += (double)__fdiv_rn(e, dc);
    }
  }
  double ray[3] = {acc[0], acc[1], 0.0};
  block_reduce(ray, err);
  __syncthreads();
  double ch[3] = {0.0, 0.0, 0.0};   // Σ pred -> GT, Σ GT -> pred squared NN distances
  int unused = 0;
  if (A.cham_fwd) {
    for (int j = threadIdx.x; j < n_pin; j += kErrThreads) ch[0] += (double)A.cham_fwd[(size_t)s * A.Mp + j];
    for (int j = threadIdx.x; j < n_gin; j += kErrThreads) ch[1] += (double)A.cham_bwd[(size_t)s * A.Mg + j];
  }
  block_reduce(ch, unused);
  if (threadIdx.x == 0) {
    // compute_chamfer_distance_inner: 0.0 when either side is empty, else the fp32 mean of both directions
    float cham = 0.f;
    if (n_pin > 0 && n_gin > 0)
      cham = __fdiv_rn(__fadd_rn(__fdiv_rn((float)ch[0], (float)n_pin), __fdiv_rn((float)ch[1], (float)n_gin)), 2.f);
    // compute_ray_errors: sums over the valid rays / count (the GT rays with d > 1e-2); 0 / 0 = NaN
    float l1 = __fdiv_rn((float)ray[0], (float)n_gsph), absrel = __fdiv_rn((float)ray[1], (float)n_gsph);
    if (n_psph == 0 && n_gsph > 0) l1 = absrel = NAN;      // no predicted ray to interpolate from
    double* out = A.out + (size_t)s * 4;
    out[0] = cham;
    out[1] = l1;
    out[2] = absrel;
    out[3] = err & 1 ? -1.0 : (err & 2 ? -2.0 : (double)n_gsph);
  }
}

}  // namespace
}  // namespace vidar

using namespace vidar;

extern "C" int vidar_eval_gather(const float* origin, const float* points, const float* tindex, const float* gt_dist,
                                 const float* pred_dist, const float* pc_range_host, int within_grid, float* pred_in,
                                 float* gt_in, float* pred_sph, float* pred_dhat, float* gt_sph, float* gt_pts,
                                 int64_t* counts, int bs, int M, int F, void* stream) {
  VIDAR_REQUIRE(origin && points && tindex && pc_range_host && pred_in && gt_in && pred_sph && pred_dhat && gt_sph &&
                    gt_pts && counts, "eval_gather: null pointer argument");
  VIDAR_REQUIRE((gt_dist == nullptr) == (pred_dist == nullptr), "eval_gather: gt_dist and pred_dist go together");
  VIDAR_REQUIRE(bs > 0 && M > 0 && F > 0 && (long long)bs * F <= 2147483647LL, "eval_gather: bad sizes bs=%d M=%d F=%d",
                bs, M, F);
  GatherArgs A;
  A.origin = origin; A.points = points; A.tindex = tindex; A.gt_dist = gt_dist; A.pred_dist = pred_dist;
  for (int i = 0; i < 6; ++i) A.range[i] = pc_range_host[i];
  A.within = within_grid; A.M = M; A.F = F;
  A.pred_in = pred_in; A.gt_in = gt_in; A.pred_sph = pred_sph; A.pred_dhat = pred_dhat; A.gt_sph = gt_sph;
  A.gt_pts = gt_pts; A.counts = counts;
  eval_gather_kernel<<<(unsigned)(bs * F), kGatherThreads, 0, (cudaStream_t)stream>>>(A);
  return check_launch("eval_gather");
}

extern "C" int vidar_eval_ray_errors(const float* origin, const float* pred_dhat, const float* gt_pts,
                                     const int64_t* nn_idx, const float* cham_fwd, const float* cham_bwd,
                                     const int64_t* counts, double* out, int N, int Mp, int Mg, void* stream) {
  VIDAR_REQUIRE(origin && pred_dhat && gt_pts && nn_idx && counts && out, "eval_ray_errors: null pointer argument");
  VIDAR_REQUIRE((cham_fwd == nullptr) == (cham_bwd == nullptr), "eval_ray_errors: cham_fwd and cham_bwd go together");
  VIDAR_REQUIRE(N > 0 && Mp > 0 && Mg > 0, "eval_ray_errors: bad sizes N=%d Mp=%d Mg=%d", N, Mp, Mg);
  ErrArgs A;
  A.origin = origin; A.pred_dhat = pred_dhat; A.gt_pts = gt_pts; A.cham_fwd = cham_fwd; A.cham_bwd = cham_bwd;
  A.nn_idx = nn_idx; A.counts = counts; A.out = out; A.Mp = Mp; A.Mg = Mg;
  eval_ray_errors_kernel<<<(unsigned)N, kErrThreads, 0, (cudaStream_t)stream>>>(A);
  return check_launch("eval_ray_errors");
}
