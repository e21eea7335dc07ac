// On-device trajectory composition and KITTI relative-trajectory-error evaluation (SURVEY 8f-4).
//
//   pose_rel_kernel      : [N,2,6] pose vectors -> the relative 4x4 motions the reference's CLI composes
//                          (test_kitti_pose.py:136-145; pose_vec2mat = utils/geo_utils.py:12-63, 93-119 in fp32,
//                          the inverse of tgt->src1 in fp64)
//   traj_scan_kernel     : P_0 = I, P_{i+1} = P_i . rel_i (test_kitti_pose.py:147-149) as a three-phase blocked
//                          prefix product in fp64 (chunk-local products, a scan of the chunk totals, fix-up)
//   kitti_dist_kernel    : trajectoryDistances (kitti_benchmark/cpp/test_odometry_all.cpp:44-56): the devkit
//                          accumulates in FLOAT, sequentially -- one thread does exactly that, so that
//                          lastFrameFromSegmentLength picks the same frames
//   kitti_segments_kernel: calcSequenceErrors (:80-125): one thread per (first_frame, length)
//   kitti_stats_kernel   : saveStats: mean t_err, r_err over the valid segments (fixed order)
// Everything is HBM-trivial (a 4541-frame sequence is 0.6 MB): the point is that a sweep over many sequences /
// checkpoints never leaves the device, not bandwidth.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace davo {

struct Mat4 { double m[16]; };

__device__ __forceinline__ void mat4_identity(double* a) {
#pragma unroll
  for (int i = 0; i < 16; ++i) a[i] = (i % 5 == 0) ? 1.0 : 0.0;
}
__device__ __forceinline__ void mat4_mul(const double* a, const double* b, double* c) {   // c = a . b (c may not alias)
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < 4; ++k) s += a[i * 4 + k] * b[k * 4 + j];
      c[i * 4 + j] = s;
    }
}
// General 4x4 inverse, Gauss-Jordan with partial pivoting (what Matrix::inv / LAPACK do; the matrices here are
// rigid motions up to rounding, so no pivot is ever small).
__device__ __forceinline__ void mat4_inv(const double* a, double* out) {
  double w[4][8];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) { w[i][j] = a[i * 4 + j]; w[i][4 + j] = i == j ? 1.0 : 0.0; }
  for (int c = 0; c < 4; ++c) {
    int piv = c;
    for (int r = c + 1; r < 4; ++r) if (fabs(w[r][c]) > fabs(w[piv][c])) piv = r;
    if (piv != c) for (int j = 0; j < 8; ++j) { const double t = w[c][j]; w[c][j] = w[piv][j]; w[piv][j] = t; }
    const double inv = 1.0 / w[c][c];
    for (int j = 0; j < 8; ++j) w[c][j] *= inv;
    for (int r = 0; r < 4; ++r) if (r != c) {
      const double f = w[r][c];
      for (int j = 0; j < 8; ++j) w[r][j] -= f * w[c][j];
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) out[i * 4 + j] = w[i][4 + j];
}

// utils/geo_utils.py:12-63, 105-119 in fp32 like the TF graph: angles clipped to [-pi, pi], R = Rx . Ry . Rz of
// [rz, ry, rx], T = [R t; 0 0 0 1].  The two matrix products are evaluated in the reference's order.
__device__ __forceinline__ void pose_vec2mat_f32(const float* v, double* out) {
  const float pi = 3.14159265358979323846f;
  const float z = fminf(fmaxf(v[0], -pi), pi), y = fminf(fmaxf(v[1], -pi), pi), x = fminf(fmaxf(v[2], -pi), pi);
  const float cz = cosf(z), sz = sinf(z), cy = cosf(y), sy = sinf(y), cx = cosf(x), sx = sinf(x);
  const float Z[9] = {cz, -sz, 0.f, sz, cz, 0.f, 0.f, 0.f, 1.f};
  const float Y[9] = {cy, 0.f, sy, 0.f, 1.f, 0.f, -sy, 0.f, cy};
  const float X[9] = {1.f, 0.f, 0.f, 0.f, cx, -sx, 0.f, sx, cx};
  float XY[9], R[9];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      float s = 0.f;
#pragma unroll
      for (int k = 0; k < 3; ++k) s = __fmaf_rn(X[i * 3 + k], Y[k * 3 + j], s);
      XY[i * 3 + j] = s;
    }
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      float s = 0.f;
#pragma unroll
      for (int k = 0; k < 3; ++k) s = __fmaf_rn(XY[i * 3 + k], Z[k * 3 + j], s);
      R[i * 3 + j] = s;
    }
#pragma unroll
  for (int i = 0; i < 3; ++i) {
#pragma unroll
    for (int j = 0; j < 3; ++j) out[i * 4 + j] = (double)R[i * 3 + j];
    out[i * 4 + 3] = (double)v[3 + i];
  }
  out[12] = 0.0; out[13] = 0.0; out[14] = 0.0; out[15] = 1.0;
}

// rel[0] = T(pose[0,0]) (the poses start at sample 0 of a sequence), then rel[1 + s] = inv(T(pose[s,1]))
// (test_kitti_pose.py:143-145, batch_size 1)
__global__ void __launch_bounds__(128) pose_rel_kernel(const float* __restrict__ poses, int n, Mat4* __restrict__ rel) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n + 1) return;
  double t[16];
  if (i == 0) {
    pose_vec2mat_f32(poses, rel[0].m);
  } else {
    pose_vec2mat_f32(poses + (size_t)(i - 1) * 12 + 6, t);
    mat4_inv(t, rel[i].m);
  }
}

// The online form of the chain (davo_odometry_push): P <- P . rel[i] for i < m in frame order, traj[first + i] = P; with
// `first` the chain starts from P_0 = I (also written to traj[0]) instead of the carried *P, which receives the last P.
// One whole warp: lane l < 16 owns element l of P and sums its row-by-column product in k = 0..3 order, as mat4_mul
// does, so that the result does not depend on how the frames were cut into pushes; P[r][k] comes from its owner by
// shuffle.  Every push runs this code (odometry_many.cuh: odo_compose_many_kernel).
__device__ __forceinline__ void traj_chain(const Mat4* rel, int m, int first, double* P, Mat4* traj) {
  const int lane = threadIdx.x & 31, l = lane & 15, r = l >> 2, c = l & 3;
  const bool owner = lane < 16;
  double p = first ? (l % 5 == 0 ? 1.0 : 0.0) : P[l];
  if (first && owner) traj[0].m[l] = p;
  for (int i = 0; i < m; ++i) {
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < 4; ++k) s += __shfl_sync(0xffffffffu, p, r * 4 + k) * rel[i].m[k * 4 + c];
    p = s;
    if (owner) traj[first + i].m[l] = p;
  }
  if (owner) P[l] = p;
}

// traj[0] = I, traj[i + 1] = traj[i] . rel[i], i < m.  One block; thread t owns elements [t*chunk, (t+1)*chunk).
__global__ void __launch_bounds__(256) traj_scan_kernel(const Mat4* __restrict__ rel, int m, int chunk, Mat4* __restrict__ traj) {
  extern __shared__ double sh[];                     // [blockDim][16] chunk totals, then their exclusive prefixes
  const int t = threadIdx.x;
  const int lo = t * chunk, hi = min(lo + chunk, m);
  double acc[16], tmp[16];
  mat4_identity(acc);
  for (int i = lo; i < hi; ++i) {                    // phase 1: local inclusive products, stored in place of the result
    mat4_mul(acc, rel[i].m, tmp);
#pragma unroll
    for (int k = 0; k < 16; ++k) { acc[k] = tmp[k]; traj[i + 1].m[k] = tmp[k]; }
  }
#pragma unroll
  for (int k = 0; k < 16; ++k) sh[t * 16 + k] = acc[k];
  __syncthreads();
  if (t == 0) {                                      // phase 2: exclusive scan of the totals, in order
    double run[16];
    mat4_identity(run);
    for (int j = 0; j < (int)blockDim.x; ++j) {
      double tot[16];
#pragma unroll
      for (int k = 0; k < 16; ++k) { tot[k] = sh[j * 16 + k]; sh[j * 16 + k] = run[k]; }
      mat4_mul(run, tot, tmp);
#pragma unroll
      for (int k = 0; k < 16; ++k) run[k] = tmp[k];
    }
    mat4_identity(traj[0].m);
  }
  __syncthreads();
  if (t > 0) {                                       // phase 3: left-multiply by the prefix of the chunks before
    double pre[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) pre[k] = sh[t * 16 + k];
    for (int i = lo; i < hi; ++i) {
      double cur[16];
#pragma unroll
      for (int k = 0; k < 16; ++k) cur[k] = traj[i + 1].m[k];
      mat4_mul(pre, cur, tmp);
#pragma unroll
      for (int k = 0; k < 16; ++k) traj[i + 1].m[k] = tmp[k];
    }
  }
}

// ---- KITTI devkit (kitti_benchmark/cpp/test_odometry_all.cpp) ------------------------------------------------
constexpr int kKittiLengths = 8;                      // {100, ..., 800} m (:13-14)
constexpr int kKittiStep = 10;                        // first frames every 10 frames (:86)

__global__ void kitti_dist_kernel(const Mat4* __restrict__ gt, int n, float* __restrict__ dist) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  float d = 0.f;
  dist[0] = 0.f;
  for (int i = 1; i < n; ++i) {                       // :44-56, float accumulation in frame order
    const float dx = (float)(gt[i - 1].m[3] - gt[i].m[3]);
    const float dy = (float)(gt[i - 1].m[7] - gt[i].m[7]);
    const float dz = (float)(gt[i - 1].m[11] - gt[i].m[11]);
    d = d + sqrtf(dx * dx + dy * dy + dz * dz);
    dist[i] = d;
  }
}

struct KittiSeg { int first_frame, last_frame; float r_err, t_err, len, speed; };

__global__ void __launch_bounds__(128) kitti_segments_kernel(const Mat4* __restrict__ gt, const Mat4* __restrict__ res, const float* __restrict__ dist,
                                                            int n, int n_first, KittiSeg* __restrict__ out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_first * kKittiLengths) return;
  const int ff = (idx / kKittiLengths) * kKittiStep, li = idx % kKittiLengths;
  const float len = 100.f * (float)(li + 1);
  KittiSeg s;
  s.first_frame = ff; s.last_frame = -1; s.r_err = 0.f; s.t_err = 0.f; s.len = len; s.speed = 0.f;
  // lastFrameFromSegmentLength (:58-63): the first i >= ff with dist[i] > dist[ff] + len (dist is non-decreasing)
  const float thr = dist[ff] + len;
  int lo = ff, hi = n;                                // first index in [lo, hi) whose dist exceeds thr
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (dist[mid] > thr) hi = mid; else lo = mid + 1;
  }
  if (lo < n) {
    const int lf = lo;
    double a[16], dg[16], dr[16], e[16];
    mat4_inv(gt[ff].m, a);  mat4_mul(a, gt[lf].m, dg);             // :104
    mat4_inv(res[ff].m, a); mat4_mul(a, res[lf].m, dr);            // :105
    mat4_inv(dr, a);        mat4_mul(a, dg, e);                    // :106
    const float ta = (float)e[0], tb = (float)e[5], tc = (float)e[10];
    const float d = (float)(0.5 * ((double)(ta + tb + tc) - 1.0));          // rotationError (:65-71): float a+b+c, double 0.5*(..-1.0), to float
    const float r_err = acosf(fmaxf(fminf(d, 1.0f), -1.0f));
    const float dx = (float)e[3], dy = (float)e[7], dz = (float)e[11];
    const float t_err = sqrtf(dx * dx + dy * dy + dz * dz);       // translationError (:73-78)
    const float num_frames = (float)(lf - ff + 1);
    s.last_frame = lf; s.r_err = r_err / len; s.t_err = t_err / len;
    s.speed = (float)((double)len / (0.1 * (double)num_frames));  // :113-114
  }
  out[idx] = s;
}

// saveStats: t_err / num, r_err / num over the segments that exist, accumulated in float in segment order
__global__ void kitti_stats_kernel(const KittiSeg* __restrict__ seg, int count, float* __restrict__ out3) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  float t = 0.f, r = 0.f, num = 0.f;
  for (int i = 0; i < count; ++i)
    if (seg[i].last_frame >= 0) { t += seg[i].t_err; r += seg[i].r_err; num += 1.f; }
  out3[0] = num > 0.f ? t / num : 0.f;
  out3[1] = num > 0.f ? r / num : 0.f;
  out3[2] = num;
}

}  // namespace davo
