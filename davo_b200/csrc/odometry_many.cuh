// Batched odometry pushes (include/davo_b200.h: davo_odometry_push_many): the kernels around the forward.
//
//   odo_stage_kernel        : every sample of the call into one stacked-triplet staging batch (input_view.cuh:
//                             stacked_view), each frame slot from the session's carried state or the caller's buffer,
//                             only the planes the sample's pair selection reads; labels become bytes on the way
//   odo_carry_kernel        : each session's new carried state (last two frames, the flow_fwd entry a later sample
//                             reads) from its old carried state and the caller's buffers
//   odo_compose_many_kernel : one warp per session: its pose rows out of the staging poses, its relative motions and
//                             its absolute poses, chained with the code of a single push (trajectory.cuh: traj_chain)
// A push of session i is the virtual sequence of davo_odometry_push: its last `head` carried frames, then its k new
// ones; virtual frame v < head is carried frame v, else the caller's frame v - head; virtual flow entry v < fe is the
// carried flow_fwd entry, else the caller's entry v - fe.  Sample s is virtual frames (s, s+1, s+2).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "trajectory.cuh"

namespace davo {

// One session of a batched push (host-built, read by all three kernels).
struct OdoManySession {
  const uint8_t* img;                       // the caller's buffers of this push
  const float *seg, *depth, *fwd, *bwd;
  uint8_t* c_img;                           // carried state (davo_odometry: c_img, c_seg, c_depth, c_fwd, d_P)
  float *c_seg, *c_depth, *c_fwd;
  double* P;
  float* pose_out;                          // [ns,2,6]
  Mat4 *traj_out, *rel;                     // [ns + 2 first]; the session's relative-motion scratch
  int head, fe, k;
  int ns, first;                            // samples of the push; it opens the sequence (P_0 = I)
  int na, ba, bt;                           // samples s < na are staged at ba + s (both pairs), the rest at bt + s - na
  int carry_fwd;                            // the caller's flow_fwd entry that becomes the carried one, or -1
};

struct OdoStageParams {
  const OdoManySession* sess;
  const int2* smp;                          // staging sample b: (session, sample)
  long long hw;
  int na;                                   // staging samples [0, na) compute both pairs, the rest tgt -> src1 only
  int flow, labels, tgt_labels, depth;      // what the variant reads (davo_capi.cu: SeqReads)
  uint8_t* img;                             // staging batch, stacked triplets
  uint8_t* lab;
  float *dep, *fl;
};

// dst[0, bytes) = src[0, bytes), thread t of `stride`: 16-byte accesses when both ends and the length allow it
__device__ __forceinline__ void odo_copy(uint8_t* dst, const uint8_t* src, size_t bytes, size_t t, size_t stride) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src) | bytes;
  if ((a & 15) == 0) {
    const uint4* s = reinterpret_cast<const uint4*>(src);
    uint4* d = reinterpret_cast<uint4*>(dst);
    for (size_t i = t; i < bytes / 16; i += stride) d[i] = __ldg(s + i);
  } else if ((a & 3) == 0) {
    const uint32_t* s = reinterpret_cast<const uint32_t*>(src);
    uint32_t* d = reinterpret_cast<uint32_t*>(dst);
    for (size_t i = t; i < bytes / 4; i += stride) d[i] = __ldg(s + i);
  } else {
    for (size_t i = t; i < bytes; i += stride) dst[i] = __ldg(src + i);
  }
}

// The host entry points' label byte (host_convert.cpp: labels_to_bytes): the class of tf.cast(v, int32) when it is
// 0..18, else 255 (no class; NaN included).  frontend.cuh: label_at reads both forms as the same class.
__device__ __forceinline__ uint32_t odo_label_byte(float v) { return (v > -1.0f && v < 19.0f) ? (uint32_t)(int)v : 255u; }

// n float labels -> n bytes; 16 per thread step (four 16-byte loads, one 16-byte store) when aligned
__device__ __forceinline__ void odo_labels(uint8_t* dst, const float* src, size_t n, size_t t, size_t stride) {
  if (((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src) | n) & 15) == 0) {
    const float4* s = reinterpret_cast<const float4*>(src);
    uint4* d = reinterpret_cast<uint4*>(dst);
    for (size_t i = t; i < n / 16; i += stride) {
      uint32_t w[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 v = __ldg(s + 4 * i + q);
        w[q] = odo_label_byte(v.x) | odo_label_byte(v.y) << 8 | odo_label_byte(v.z) << 16 | odo_label_byte(v.w) << 24;
      }
      d[i] = make_uint4(w[0], w[1], w[2], w[3]);
    }
  } else {
    for (size_t i = t; i < n; i += stride) dst[i] = (uint8_t)odo_label_byte(__ldg(src + i));
  }
}

// grid (x, staging samples): block row b stages sample b, its blocks share each plane.  Planes a sample's selection
// does not read (src0 and flow plane 0 under tgt -> src1 only; labels per SeqReads::lab) are not written.
__global__ void __launch_bounds__(256) odo_stage_kernel(const OdoStageParams p) {
  const int b = blockIdx.y;
  const int2 m = p.smp[b];
  const OdoManySession& d = p.sess[m.x];
  const int s = m.y, head = d.head, fe = d.fe;
  const bool k0 = b < p.na;
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  const size_t hw = (size_t)p.hw;
#pragma unroll 1
  for (int j = 0; j < 3; ++j) {
    if (j == 0 && !k0) continue;                            // src0: read only by the pair tgt -> src0
    const int v = s + j;
    const bool carried = v < head;
    const size_t f = carried ? (size_t)v : (size_t)(v - head);
    const size_t slot = (size_t)b * 3 + j;
    odo_copy(p.img + slot * hw * 3, (carried ? d.c_img : d.img) + f * hw * 3, hw * 3, t, stride);
    if (p.labels && (j == 2 || j == 0 || p.tgt_labels))
      odo_labels(p.lab + slot * hw, (carried ? d.c_seg : d.seg) + f * hw, hw, t, stride);
    if (p.depth)
      odo_copy(reinterpret_cast<uint8_t*>(p.dep + slot * hw),
               reinterpret_cast<const uint8_t*>((carried ? d.c_depth : d.depth) + f * hw), hw * 4, t, stride);
  }
  if (p.flow) {
    float* dst = p.fl + (size_t)b * hw * 4;
    odo_copy(reinterpret_cast<uint8_t*>(dst + hw * 2), reinterpret_cast<const uint8_t*>(d.bwd + (size_t)(s + 1 - fe) * hw * 2),
             hw * 8, t, stride);                            // plane 1: flow_bwd entry s + 1
    if (k0)                                                 // plane 0: flow_fwd entry s
      odo_copy(reinterpret_cast<uint8_t*>(dst),
               reinterpret_cast<const uint8_t*>(s < fe ? d.c_fwd : d.fwd + (size_t)(s - fe) * hw * 2), hw * 8, t, stride);
  }
}

// carried frame c[j] (j < nc) <- virtual frame fc + j, for one plane kind of `frame` bytes per frame.  Race-free within
// the launch: c[0] may come from c[1] while c[1] takes a new frame, but element e of both is read and then written by
// the same thread only (at the same offset in each frame), and no other block or thread touches e.  Plain loads: the
// kernel writes what it reads.
template <typename T>
__device__ __forceinline__ void odo_carry_plane(uint8_t* c, const uint8_t* s0, const uint8_t* s1, int nc, size_t frame,
                                                size_t t, size_t stride) {
  T* c0 = reinterpret_cast<T*>(c);
  T* c1 = reinterpret_cast<T*>(c + frame);
  const T* a = reinterpret_cast<const T*>(s0);
  const T* b = reinterpret_cast<const T*>(s1);
  for (size_t i = t; i < frame / sizeof(T); i += stride) {
    T x{}, y{};
    if (a) x = a[i];
    if (nc > 1) y = b[i];
    if (a) c0[i] = x;
    if (nc > 1) c1[i] = y;
  }
}
__device__ __forceinline__ void odo_carry_frames(uint8_t* c, const uint8_t* carried, const uint8_t* caller, int head,
                                                 int n, size_t frame, size_t t, size_t stride) {
  const int nc = n < 2 ? n : 2, fc = n - nc;
  const uint8_t* src[2] = {nullptr, nullptr};
  for (int j = 0; j < nc; ++j) {
    const int v = fc + j;
    src[j] = v < head ? (v == j ? nullptr : carried + (size_t)v * frame) : caller + (size_t)(v - head) * frame;
  }
  const uintptr_t a = reinterpret_cast<uintptr_t>(c) | reinterpret_cast<uintptr_t>(src[0]) |
                      reinterpret_cast<uintptr_t>(src[1]) | frame;
  if ((a & 15) == 0) odo_carry_plane<uint4>(c, src[0], src[1], nc, frame, t, stride);
  else if ((a & 3) == 0) odo_carry_plane<uint32_t>(c, src[0], src[1], nc, frame, t, stride);
  else odo_carry_plane<uint8_t>(c, src[0], src[1], nc, frame, t, stride);
}

// grid (x, sessions).  Launched after odo_stage_kernel, which reads the old carried state.
__global__ void __launch_bounds__(256) odo_carry_kernel(const OdoManySession* __restrict__ sess, long long hw_, int depth) {
  const OdoManySession& d = sess[blockIdx.y];
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  const size_t hw = (size_t)hw_;
  const int n = d.head + d.k;
  odo_carry_frames(d.c_img, d.c_img, d.img, d.head, n, hw * 3, t, stride);
  if (d.c_seg)
    odo_carry_frames(reinterpret_cast<uint8_t*>(d.c_seg), reinterpret_cast<const uint8_t*>(d.c_seg),
                     reinterpret_cast<const uint8_t*>(d.seg), d.head, n, hw * 4, t, stride);
  if (depth)
    odo_carry_frames(reinterpret_cast<uint8_t*>(d.c_depth), reinterpret_cast<const uint8_t*>(d.c_depth),
                     reinterpret_cast<const uint8_t*>(d.depth), d.head, n, hw * 4, t, stride);
  if (d.carry_fwd >= 0)
    odo_copy(reinterpret_cast<uint8_t*>(d.c_fwd), reinterpret_cast<const uint8_t*>(d.fwd + (size_t)d.carry_fwd * hw * 2),
             hw * 8, t, stride);
}

// One warp per session (4 per block): pose rows, relative motions (pose_rel_kernel's formulas), the chain.
__global__ void __launch_bounds__(128) odo_compose_many_kernel(const OdoManySession* __restrict__ sess, int n,
                                                               const float* __restrict__ spose) {
  const int w = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (w >= n) return;
  const OdoManySession& d = sess[w];
  const int ns = d.ns, first = d.first;
  if (ns == 0) return;                                      // a push too short to hold a sample
  auto row = [&](int s) { return spose + (size_t)(s < d.na ? d.ba + s : d.bt + s - d.na) * 12; };
  for (int e = lane; e < ns * 12; e += 32) d.pose_out[e] = row(e / 12)[e % 12];
  for (int i = lane; i < ns + first; i += 32) {
    if (first && i == 0) {
      pose_vec2mat_f32(row(0), d.rel[0].m);
    } else {
      double t[16];
      pose_vec2mat_f32(row(i - first) + 6, t);
      mat4_inv(t, d.rel[i].m);
    }
  }
  __syncwarp();                                             // every lane's motions are visible to the chain
  traj_chain(d.rel, ns + first, first, d.P, d.traj_out);
}

}  // namespace davo
