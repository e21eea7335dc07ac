// HBM-bound front end and head of the pose path:
//   se_pool_kernel  : sum over the frame of (|.|, normalised) optical flow      (attention_module.py:66)
//   pack_kernel     : SE fully-connected layers -> 19 class weights, per-pixel
//                     class-weight gather, u8 -> [-1,1] frames, masking, and the
//                     packed PoseNN input                                       (attention_module.py:89-101,
//                                                                                davo.py:1115,1178,1404-1442,1519-1522)
//   head_kernel     : spatial mean + 1x1 pred + 0.01 scale                      (posenn.py:240-250)
// Frame pair index p = 2 * sample + source (0: tgt->src0, 1: tgt->src1), the
// row order of pred_poses (davo.py:1456-1458).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "input_view.cuh"
#include "ptx.cuh"

namespace davo {

constexpr int kPoolSplits = 16;
constexpr int kPoolDim = 24;     // >= the widest pooled vector (19 class frequencies + 2 flow means)
constexpr int kAttFrames = 4;    // attention-weight slots per unit (see unit_frame; 4: the depth-split source in a sample unit)
constexpr int kAttStride = 24;   // floats per slot of att_w: 19 class weights, or the excitation of a per-pixel source (<= 21)
constexpr int kPackedC = 16;     // widest packed PoseNN input (see pack_kernel; FrontParams::packed_c = 8 or 16)
constexpr int kNumClasses = 19;
constexpr int kPackBlocksPerPair = 104;

// Which frame pairs of a batch are computed (include/davo_b200.h: DAVO_PAIRS_*).  Slot s of the
// selection maps to (sample b, source k); the pose lands at pose_out[b][k][:].
//   0 all:              s -> (s >> 1, s & 1)
//   1 trajectory:       s -> (s, 1)            tgt->src1 only: what test_kitti_pose.py:143-145 composes
//   2 trajectory+first: 0 -> (0, 0), s -> (s - 1, 1)   plus the first sample's tgt->src0
//   3 sample units:     s -> (s, 0)            the non-shared nets take (tgt, src0, src1) at once
__host__ __device__ __forceinline__ void pair_of_slot(int mode, int s, int* b, int* k) {
  if (mode == 0) { *b = s >> 1; *k = s & 1; }
  else if (mode == 1 || mode == 3) { *b = s; *k = mode == 1 ? 1 : 0; }
  else if (s == 0) { *b = 0; *k = 0; }
  else { *b = s - 1; *k = 1; }
}

// Attention-weight slot `fr` of a unit -> frame of the sample, coded as its plane in the inputs
// (0 = src0, 1 = tgt, 2 = src1: seg[:, f], image columns [f*W, (f+1)*W); flow[:, 0] belongs to
// src0, flow[:, 1] to src1, the target's flow is zeros, davo.py:978-982).
//   frame-pair units (shared nets):  slot 0 = the pair's source frame, slot 1 = the target
//   sample units (non-shared nets):  slot 0 = src0, slot 1 = src1, slot 2 = the target
__device__ __forceinline__ int unit_frame(int unit_sample, int k, int fr) {
  if (unit_sample) return fr == 0 ? 0 : fr == 1 ? 2 : 1;
  return fr == 0 ? (k == 0 ? 0 : 2) : 1;
}

struct FrontParams {
  int H, W;
  int unit_sample;       // 1: a unit is a whole sample (tgt, src0, src1), posenn.py:12-131
  int pair0;             // first selection slot of this pass
  int pair_mode;         // see pair_of_slot
  int packed_c;          // 8: [tgt rgb, src rgb, src flow]; 16: the legacy layout of pack_kernel
  int npairs;
  int in_mode;           // 1: flows are concatenated (v1)
  int att_src;           // 0 none, 1 se_flow, 2 static, 3 se_seg, 4 se_rgb (-> seg), 5 se_depth (-> seg),
                         // 6 se_segflow (-> seg): davo.py:1117-1400
  int depth_norm;        // 1: "-norm_depth", SE depth input / 80; 2: the se_disp sources, SE input = 1 / depth of the frame
  int pool_2x2;          // se_flow only: mode='gp2x2' (attention_module.py:68-78): the means of the four
                         // quadrants [:h/2,:w/2], [:h/2,w/2:], [h/2:,:w/2], [h/2:,w/2:] concatenated -> 8 inputs
  int spp_levels;        // se_flow only: mode='spp' (attention_module.py:79-86, 137-167): pyramid levels ...
  int spp_n[3];          // ... and their out_pool_size; se_spp_kernel replaces se_pool_kernel
  int se_in, se_hid;     // SE dense sizes: in -> hid -> se_out (flow 2,8; seg 19,19; rgb 3,8)
  int depth_split;       // 1: -se_flow_on_depthseg_seplayers (davo.py:1136-1154): slot 0 / 1 of a pair hold the class weights of
  float depth_thres;     //    SE "se_flow_near" / "se_flow_far" on the SOURCE flow; a pixel reads slot 0 where depth < depth_thres
  int se_out;            // 19 class weights, or with pixel_map the excitation of the SE input itself (= se_in)
  int pixel_map;         // 1 (2: with att_src 5, depth term AND SE flow, -se_mixDepthFlow / -se_mixDispFlow, davo.py:1157-1174):
                         //    se_block sources whose map is reduce_sum(input * excitation) per pixel instead of a
                         //    class weight gathered by label (davo.py:1228-1245, 1293-1303, 1375-1379); att_src
                         //    4: r,g,b of the frame; 5: its depth term; 6: one_hot(label) and the SE flow
  int att_tgt_ones;
  int mask_rgb, mask_flow;
  int se_act;            // 0 relu, 1 tanh, 2 lrelu
  int flow_abs;          // 0 none, 1 both, 2 h, 3 v
  int flow_norm;
  InputView in;          // images, labels, depth and flow of the batch, triplet or sequence layout (input_view.cuh);
                         // the host entry points convert float labels to bytes on the CPU (in.seg8) so that a quarter
                         // of their bytes crosses PCIe
  int flow_f16;          // davo_config.flow_f16: 1 = float32 flow values are rounded to binary16 when read (flow_q)
  const float* se_w;     // W1[in][hid] b1[hid] W2[hid][19] b2[19]
  const float* static_w; // sigmoid(seg_channel_weight)[19]
  float* pool_part;      // [mb][kAttFrames][kPoolSplits][kPoolDim]
  unsigned int* pool_count;  // [mb][kAttFrames], zero between launches
  float* att_w;          // [mb][kAttFrames][kAttStride], slots as in unit_frame
  float* packed;         // [mb][H][W][packed_c]
};

// Label of pixel `pix` of plane `plane` (element offset of the plane = plane index * H*W) as the
// reference's tf.cast(seg, int32) (davo.py:1115: truncation toward zero); bytes are already ints.
// (a NaN has no class: on the CPU tf.cast gives INT_MIN for it, which one_hot turns into a zero row; CUDA's conversion
// would give 0, i.e. class "road")
__device__ __forceinline__ int label_of(float v) { return v == v ? (int)v : -1; }
__device__ __forceinline__ int label_at(const FrontParams& p, size_t plane_off, int pix) {
  if (p.in.seg8) return p.in.seg8[plane_off + pix];
  return label_of(__ldg(p.in.seg + plane_off + pix));
}
// four consecutive labels (pix % 4 == 0)
__device__ __forceinline__ void labels4_at(const FrontParams& p, size_t plane_off, int pix, int (&lab)[4]) {
  if (p.in.seg8) {
    const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(p.in.seg8 + plane_off + pix));
    lab[0] = w & 255u; lab[1] = (w >> 8) & 255u; lab[2] = (w >> 16) & 255u; lab[3] = w >> 24;
  } else {
    const float4 v = __ldg(reinterpret_cast<const float4*>(p.in.seg + plane_off + pix));
    lab[0] = label_of(v.x); lab[1] = label_of(v.y); lab[2] = label_of(v.z); lab[3] = label_of(v.w);
  }
}

// davo_config.flow_f16 = 1 (opt-in): the flow input is DEFINED as rounded to IEEE binary16 (11 significant
// bits, what the TF32 conv operands keep anyway): the host entry point can then round on the CPU and move
// half the bytes over PCIe with bit-identical results (host_convert.cpp).  Values that do not fit a finite
// half (|x| >= 65520, NaN) pass through unchanged; the host sends a chunk holding one as float32.
// Default (flow_f16 = 0): the float32 values are used as given, as the reference's graph does.
__device__ __forceinline__ float flow_q(float x) {
  return fabsf(x) < 65520.0f ? __half2float(__float2half_rn(x)) : x;
}
// two values at once: one packed f32x2 -> f16x2 conversion; a value that overflowed to infinity (or was
// not finite to begin with) is passed through, which is the same rule as flow_q
__device__ __forceinline__ float2 flow_q2(float x, float y) {
  const float2 q = __half22float2(__floats2half2_rn(x, y));
  return make_float2(fabsf(q.x) < 65520.0f ? q.x : x, fabsf(q.y) < 65520.0f ? q.y : y);
}
// pixel `pix` (x, y) of flow plane k (0: src0 -> tgt, 1: src1 -> tgt; davo.py:978-982) of sample b
__device__ __forceinline__ float2 flow1_at(const FrontParams& p, int b, int k, int pix, int hw) {
  if (b < p.in.n_flow16) {
    const __half2 h = *reinterpret_cast<const __half2*>(flow16_plane(p.in, b, k) + (size_t)pix * 2);
    return __half22float2(h);
  }
  const float2 v = __ldg(reinterpret_cast<const float2*>(flow_plane(p.in, b, k) + (size_t)pix * 2));
  return p.flow_f16 ? flow_q2(v.x, v.y) : v;
}
// pixels pix, pix + 1 (pix even): (x0, y0, x1, y1)
__device__ __forceinline__ float4 flow2_at(const FrontParams& p, int b, int k, int pix, int hw) {
  if (b < p.in.n_flow16) {
    const uint2 raw = __ldg(reinterpret_cast<const uint2*>(flow16_plane(p.in, b, k) + (size_t)pix * 2));
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&raw.x));
    const float2 c = __half22float2(*reinterpret_cast<const __half2*>(&raw.y));
    return make_float4(a.x, a.y, c.x, c.y);
  }
  const float4 v = __ldg(reinterpret_cast<const float4*>(flow_plane(p.in, b, k) + (size_t)pix * 2));
  if (!p.flow_f16) return v;
  const float2 lo = flow_q2(v.x, v.y), hi = flow_q2(v.z, v.w);
  return make_float4(lo.x, lo.y, hi.x, hi.y);
}

__device__ __forceinline__ float se_in_x(float v, const FrontParams& p) {
  if (p.flow_norm) v = (v - 0.32140523f) / 15.384229f;
  if (p.flow_abs == 1 || p.flow_abs == 2) v = fabsf(v);
  return v;
}
__device__ __forceinline__ float se_in_y(float v, const FrontParams& p) {
  if (p.flow_norm) v = (v - 0.32140523f) / 15.384229f;
  if (p.flow_abs == 1 || p.flow_abs == 3) v = fabsf(v);
  return v;
}
__device__ __forceinline__ float se_activation(float v, int act) {
  if (act == 1) return tanhf(v);
  if (act == 2) return v > 0.f ? v : 0.2f * v;
  return fmaxf(v, 0.f);
}

// The two dense layers of se() / se_block() (attention_module.py:89-101 / :37-50) on a pooled vector held in
// shared memory: s_pool[D] -> activation(W1 . + b1)[hid] -> sigmoid(W2 . + b2)[se_out] -> att_w[pl][fr][:].  Called by
// a whole 256-thread block after a barrier that made s_pool visible; p.se_w = W1[D][hid] b1[hid] W2[hid][out] b2[out].
__device__ __forceinline__ void se_dense_layers(const FrontParams& p, const float* s_pool, float* s_fc1, int D,
                                                int pl, int fr) {
  const int Hd = p.se_hid;
  // depth_split: slot fr uses its own weight set (near, far), stored one after the other
  const int wset = p.unit_sample ? (fr & 1) : fr;           // sample units: slots (0,1) / (2,3) = (near, far) of src0 / src1
  const float* W1 = p.se_w + (p.depth_split ? wset * (D * Hd + Hd + Hd * p.se_out + p.se_out) : 0);
  const float* b1 = W1 + D * Hd;
  const float* W2 = b1 + Hd;
  const int out = p.se_out;
  const float* b2 = W2 + Hd * out;
  if (threadIdx.x < Hd) {
    float a = b1[threadIdx.x];
    for (int i = 0; i < D; ++i) a += s_pool[i] * W1[i * Hd + threadIdx.x];
    s_fc1[threadIdx.x] = se_activation(a, p.se_act);
  }
  __syncthreads();
  if (threadIdx.x < out) {
    const int c = threadIdx.x;
    float a = b2[c];
    for (int j = 0; j < Hd; ++j) a += s_fc1[j] * W2[j * out + c];
    p.att_w[((size_t)pl * kAttFrames + fr) * kAttStride + c] = 1.0f / (1.0f + expf(-a));
  }
}

// grid (kPoolSplits, npairs, frames), 256 threads.  Global average pool of the SE input in
// deterministic partial sums (attention_module.py:66 / :22); the block that finishes a
// (pair, frame) last adds the partials in a fixed order and runs the two dense layers
// (attention_module.py:89-101 / :37-50) -> att_w[pair][frame][19].
//   se_flow (davo.py:1176):      pool = mean of the (abs / normalised) flow, 2 -> 8 -> 19
//   se_seg (davo.py:1306, 1313): pool = class frequencies of one_hot(label) (out-of-range labels
//                                 are all-zero rows), 19 -> 19 -> 19; excitation * one_hot summed
//                                 over classes = excitation[label]
//   se_rgb*_to_seg (davo.py:1277, 1287): pool = mean r, g, b of the frame, 3 -> 8 -> 19
//   se_depth*_to_seg (davo.py:1214, 1223): pool = mean(depth of the frame + depth of the TARGET):
//                                 davo.py:1109 adds a Tensor to a Python list, which TensorFlow
//                                 broadcasts ([d_tgt, d_src0, d_src1] + d_tgt); 1 -> 8 -> 19
//   se_SegFlow_to_seg* (davo.py:1341-1372): pool of concat(one_hot(label), SE flow) = the 19 class
//                                 frequencies followed by the 2 flow means, 21 -> 19|8 -> 19; the
//                                 target's flow is zeros, whose SE input is the constant se_in(0)
// blockIdx.z = 0: the pair's source frame; 1: the target frame (variants that do not force the
// target map to ones).
// The body of se_pool_kernel for block (split bx, unit pl, slot fr); returns true in the one block that finished the
// (unit, slot) and wrote its class weights.  Also called by front_pipeline_kernel.
__device__ __forceinline__ bool se_pool_body(const FrontParams& p, const int bx, const int pl, const int fr) {
  int b, k;
  pair_of_slot(p.pair_mode, p.pair0 + pl, &b, &k);
  const int hw = p.H * p.W;
  const int D = p.se_in;
  // depth_split: a source frame has two slots (near, far), both pooling that frame's flow: slots (0, 1) of a frame pair;
  // (0, 1) = src0 and (2, 3) = src1 of a sample unit
  const int f = unit_frame(p.unit_sample, k, p.depth_split ? (p.unit_sample ? (fr >> 1) : 0) : fr);
  __shared__ float red[8][4];
  __shared__ int s_hist[kNumClasses];
  __shared__ float s_pool[kPoolDim];
  __shared__ float s_fc1[kPoolDim];
  __shared__ int s_last;
  float* part = p.pool_part + (((size_t)pl * kAttFrames + fr) * kPoolSplits + bx) * kPoolDim;
  if (p.att_src == 3 || p.att_src == 6) {
    if (threadIdx.x < kNumClasses) s_hist[threadIdx.x] = 0;
    __syncthreads();
    const size_t seg_off = frame_plane(p.in, b, f, hw);
    const int per = (hw + kPoolSplits - 1) / kPoolSplits;
    const int beg = bx * per, end = min(beg + per, hw);
    for (int i = beg + threadIdx.x; i < end; i += 256) {
      const int lab = label_at(p, seg_off, i);                   // tf.cast truncates toward zero
      if (lab >= 0 && lab < kNumClasses) atomicAdd(&s_hist[lab], 1);   // integer counts: exact, order-free
    }
    __syncthreads();
    if (threadIdx.x < kNumClasses) part[threadIdx.x] = (float)s_hist[threadIdx.x];
    if (p.att_src == 6) {                       // + the flow sums of this split -> part[19], part[20]
      float s0 = 0.f, s1 = 0.f;
      if (f != 1) {
        const int n4 = hw / 2;
        const int per4 = (n4 + kPoolSplits - 1) / kPoolSplits;
        const int beg4 = bx * per4, end4 = min(beg4 + per4, n4);
        for (int i = beg4 + threadIdx.x; i < end4; i += 256) {
          const float4 v = flow2_at(p, b, f == 2 ? 1 : 0, 2 * i, hw);
          s0 += se_in_x(v.x, p) + se_in_x(v.z, p);
          s1 += se_in_y(v.y, p) + se_in_y(v.w, p);
        }
      }
#pragma unroll
      for (int o = 16; o >= 1; o >>= 1) {
        s0 += __shfl_xor_sync(0xffffffffu, s0, o);
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      }
      if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5][0] = s0; red[threadIdx.x >> 5][1] = s1; }
      __syncthreads();
      if (threadIdx.x < 2) {
        float a = 0.f;
        for (int i = 0; i < 8; ++i) a += red[i][threadIdx.x];
        part[kNumClasses + threadIdx.x] = a;
      }
    }
  } else {
    float s0 = 0.f, s1 = 0.f, s2 = 0.f;
    if (p.att_src == 5) {
      const float4* df = reinterpret_cast<const float4*>(p.in.depth + frame_plane(p.in, b, f, hw));
      const float4* dt = reinterpret_cast<const float4*>(p.in.depth + frame_plane(p.in, b, 1, hw));
      const int n4 = hw / 4;
      const int per = (n4 + kPoolSplits - 1) / kPoolSplits;
      const int beg = bx * per, end = min(beg + per, n4);
      if (p.depth_norm == 2)                          // se_disp*_to_seg (davo.py:1253-1270): 1. / depth, no target term
        for (int i = beg + threadIdx.x; i < end; i += 256) {
          const float4 a = __ldg(df + i);
          s0 += 1.0f / a.x + 1.0f / a.y + 1.0f / a.z + 1.0f / a.w;
        }
      else
      for (int i = beg + threadIdx.x; i < end; i += 256) {
        const float4 a = __ldg(df + i), c = __ldg(dt + i);
        s0 += (a.x + c.x) + (a.y + c.y) + (a.z + c.z) + (a.w + c.w);
      }
      if (p.pixel_map == 2 && f != 1)                 // -se_mixDepthFlow / -se_mixDispFlow: + the two SE flow means
        for (int i = beg + threadIdx.x; i < end; i += 256) {
          const float4 v0 = flow2_at(p, b, f == 2 ? 1 : 0, 4 * i, hw), v1 = flow2_at(p, b, f == 2 ? 1 : 0, 4 * i + 2, hw);
          s1 += se_in_x(v0.x, p) + se_in_x(v0.z, p) + se_in_x(v1.x, p) + se_in_x(v1.z, p);
          s2 += se_in_y(v0.y, p) + se_in_y(v0.w, p) + se_in_y(v1.y, p) + se_in_y(v1.w, p);
        }
    } else if (p.att_src == 1) {
      const int fk = f == 2 ? 1 : 0;                  // flow plane of this frame
      const int n4 = hw / 2;                          // one load = 2 pixels
      const int per = (n4 + kPoolSplits - 1) / kPoolSplits;
      const int beg = bx * per, end = min(beg + per, n4);
      if (f != 1 && !p.pool_2x2)                      // the target's flow is all zeros (davo.py:979)
#pragma unroll 4                                      // four loads in flight per thread; the sums keep their order
        for (int i = beg + threadIdx.x; i < end; i += 256) {
          const float4 v = flow2_at(p, b, fk, 2 * i, hw);
          s0 += se_in_x(v.x, p) + se_in_x(v.z, p);
          s1 += se_in_y(v.y, p) + se_in_y(v.w, p);
        }
      if (f != 1 && p.pool_2x2) {
        // per-quadrant sums: this thread's 8 accumulators, reduced over the block into part[0..7]
        float q[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        const int hh = p.H / 2, hw2 = p.W / 2;
        for (int i = beg + threadIdx.x; i < end; i += 256) {
          const float4 v = flow2_at(p, b, fk, 2 * i, hw);
          const int pix = 2 * i, h = pix / p.W, w = pix - h * p.W;       // W is even: both pixels in one row
          const int qa = (h >= hh ? 2 : 0) + (w >= hw2 ? 1 : 0), qb = (h >= hh ? 2 : 0) + (w + 1 >= hw2 ? 1 : 0);
#pragma unroll
          for (int k2 = 0; k2 < 4; ++k2) {
            if (qa == k2) { q[2 * k2] += se_in_x(v.x, p); q[2 * k2 + 1] += se_in_y(v.y, p); }
            if (qb == k2) { q[2 * k2] += se_in_x(v.z, p); q[2 * k2 + 1] += se_in_y(v.w, p); }
          }
        }
        __shared__ float red8[8][8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
#pragma unroll
          for (int o = 16; o >= 1; o >>= 1) q[j] += __shfl_xor_sync(0xffffffffu, q[j], o);
          if ((threadIdx.x & 31) == 0) red8[threadIdx.x >> 5][j] = q[j];
        }
        __syncthreads();
        if (threadIdx.x < 8) {
          float a = 0.f;
          for (int i = 0; i < 8; ++i) a += red8[i][threadIdx.x];
          part[threadIdx.x] = a;
        }
        __syncthreads();
      }
    } else {
      // byte sums are exact; the affine map to [-1, 1] (davo.py:1519-1522) is applied to the mean
      const uint8_t* img_f = frame_img(p.in, b, f);
      const int per = (hw + kPoolSplits - 1) / kPoolSplits;
      const int beg = bx * per, end = min(beg + per, hw);
      unsigned int u0 = 0, u1 = 0, u2 = 0;
      for (int i = beg + threadIdx.x; i < end; i += 256) {
        const int h = i / p.W, w = i - h * p.W;
        const uint8_t* px = img_f + (size_t)h * p.in.img_row + w * 3;
        u0 += px[0]; u1 += px[1]; u2 += px[2];
      }
      s0 = (float)u0; s1 = (float)u1; s2 = (float)u2;
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
      s0 += __shfl_xor_sync(0xffffffffu, s0, o);
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    if ((threadIdx.x & 31) == 0) {
      red[threadIdx.x >> 5][0] = s0; red[threadIdx.x >> 5][1] = s1; red[threadIdx.x >> 5][2] = s2;
    }
    __syncthreads();
    if (threadIdx.x < 3 && !(p.att_src == 1 && p.pool_2x2 && f != 1)) {
      float a = 0.f;
      for (int i = 0; i < 8; ++i) a += red[i][threadIdx.x];
      part[threadIdx.x] = a;
    }
    if (p.att_src == 1 && p.pool_2x2 && f == 1 && threadIdx.x >= 3 && threadIdx.x < 8) part[threadIdx.x] = 0.f;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned int done = atomicAdd(&p.pool_count[pl * kAttFrames + fr], 1u);
    s_last = (done == kPoolSplits - 1);
    if (s_last) p.pool_count[pl * kAttFrames + fr] = 0;       // ready for the next launch
  }
  __syncthreads();
  if (!s_last) return false;
  __threadfence();
  if (threadIdx.x < D) {
    const float* pp = p.pool_part + ((size_t)pl * kAttFrames + fr) * kPoolSplits * kPoolDim + threadIdx.x;
    float a = 0.f;
    for (int sp = 0; sp < kPoolSplits; ++sp) a += __ldcg(pp + sp * kPoolDim);
    if (p.att_src == 1 && p.pool_2x2) {            // quadrant pixel counts (attention_module.py:70-71: h//2, w//2)
      const int qd = threadIdx.x >> 1;
      const int rows = (qd & 2) ? p.H - p.H / 2 : p.H / 2, cols = (qd & 1) ? p.W - p.W / 2 : p.W / 2;
      a *= 1.0f / (float)(rows * cols);
    } else {
      a *= 1.0f / (float)hw;
    }
    if (p.att_src == 6 && f == 1 && threadIdx.x >= kNumClasses)      // mean of a constant map: the target's zero flow
      a = threadIdx.x == kNumClasses ? se_in_x(0.f, p) : se_in_y(0.f, p);
    if (p.att_src == 4) a = a * (1.0f / 255.0f) * 2.0f - 1.0f;
    if (p.att_src == 5 && p.depth_norm == 1 && threadIdx.x == 0) a = a / 80.0f;
    if (p.att_src == 5 && f == 1 && threadIdx.x >= 1)                // depth + flow sources: the target's zero flow
      a = threadIdx.x == 1 ? se_in_x(0.f, p) : se_in_y(0.f, p);
    s_pool[threadIdx.x] = a;
  }
  __syncthreads();
  se_dense_layers(p, s_pool, s_fc1, D, pl, fr);
  return true;
}

__global__ void __launch_bounds__(256) se_pool_kernel(const FrontParams p) {
  pdl_launch_dependents();
  pdl_wait();                     // workspace buffers are shared with the kernels before this one
  se_pool_body(p, blockIdx.x, blockIdx.y, blockIdx.z);
}

// se(flow, "se_flow", [8,19], mode='spp', spp_size) (davo.py:1193-1210): spatial_pyramid_pool
// (attention_module.py:137-167) as TensorFlow evaluates it.  Per level n: h_size = ceil(H/n), w_size =
// ceil(W/n); the SE flow is zero-padded (bottom / right) to n*h_size x n*w_size, then avg_pool with a window of
// h_size x H_SIZE -- the reference passes h_size for both sides (:158) -- at strides (h_size, w_size), 'SAME'.
// For H <= W the window is narrower than the stride, 'SAME' pads nothing, and cell (i, j) is the mean over
// rows [i*h_size, (i+1)*h_size) x columns [j*w_size, j*w_size + h_size) with the tf.pad zeros counted: only the
// left part of each cell is read.  Pooled vector: levels concatenated, cells row-major, (x, y) last.
// grid (npairs, source frames), 256 threads: a warp per cell, then the two dense layers -> att_w.
constexpr int kSppMaxDim = 232;                          // (64 + 36 + 16) cells x 2
__global__ void __launch_bounds__(256) se_spp_kernel(const FrontParams p) {
  pdl_launch_dependents();
  pdl_wait();
  const int pl = blockIdx.x, fr = blockIdx.y;
  int b, k;
  pair_of_slot(p.pair_mode, p.pair0 + pl, &b, &k);
  const int hw = p.H * p.W;
  const int f = unit_frame(p.unit_sample, k, fr);
  const int fk = f == 2 ? 1 : 0;                        // flow plane of this frame (never the target here)
  __shared__ float s_pool[kSppMaxDim];
  __shared__ float s_fc1[kPoolDim];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int cell0 = 0;
  for (int lv = 0; lv < p.spp_levels; ++lv) {
    const int n = p.spp_n[lv];
    const int hs = (p.H + n - 1) / n, ws = (p.W + n - 1) / n;
    const float inv = 1.0f / (float)(hs * hs);
    for (int cell = warp; cell < n * n; cell += 8) {
      const int y0 = (cell / n) * hs, x0 = (cell % n) * ws;
      float sx = 0.f, sy = 0.f;
      for (int i = lane; i < hs * hs; i += 32) {
        const int y = y0 + i / hs, x = x0 + i % hs;
        if (y < p.H && x < p.W) {                       // beyond the map: tf.pad zeros
          const float2 v = flow1_at(p, b, fk, y * p.W + x, hw);
          sx += se_in_x(v.x, p);
          sy += se_in_y(v.y, p);
        }
      }
#pragma unroll
      for (int o = 16; o >= 1; o >>= 1) {
        sx += __shfl_xor_sync(0xffffffffu, sx, o);
        sy += __shfl_xor_sync(0xffffffffu, sy, o);
      }
      if (lane == 0) { s_pool[(cell0 + cell) * 2] = sx * inv; s_pool[(cell0 + cell) * 2 + 1] = sy * inv; }
    }
    cell0 += n * n;
  }
  __syncthreads();
  se_dense_layers(p, s_pool, s_fc1, cell0 * 2, pl, fr);
}

// se_block(seg_19, "se_seg", ratio=1, mode='gp2x2') (davo.py:1317-1322) and se_spp_block(seg_19, "se_spp_seg",
// ratio=1, spp_size) (davo.py:1323-1340; attention_module.py:105-135): the one-hot label map pooled per cell --
// the four quadrants [:h/2,:w/2] ... [h/2:,w/2:] (attention_module.py:26-35), or the pyramid cells of
// se_spp_kernel (left h_size x h_size square of every cell, tf.pad zeros counted) -- i.e. the class
// frequencies of each cell, 19 per cell, then dense -> 19 (activation) -> 19 (sigmoid); the map is
// excitation[label].  grid (npairs, frames), 256 threads: a warp per cell with a shared-memory histogram.
constexpr int kSegCellsMaxDim = (64 + 36 + 16) * kNumClasses;      // 2204
__global__ void __launch_bounds__(256) se_segcells_kernel(const FrontParams p) {
  pdl_launch_dependents();
  pdl_wait();
  const int pl = blockIdx.x, fr = blockIdx.y;
  int b, k;
  pair_of_slot(p.pair_mode, p.pair0 + pl, &b, &k);
  const int hw = p.H * p.W;
  const int f = unit_frame(p.unit_sample, k, fr);
  const size_t seg_off = frame_plane(p.in, b, f, hw);
  __shared__ float s_pool[kSegCellsMaxDim];
  __shared__ int s_hist[8][kNumClasses];
  __shared__ float s_fc1[kPoolDim];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int cell0 = 0;
  const int levels = p.pool_2x2 ? 1 : p.spp_levels;
  // -se_spp21_mixSegFlow (davo.py:1380-1383): the pooled map is concat(one_hot(label), SE flow): 19 + 2 values per cell
  const bool with_flow = p.att_src == 6;
  const int cs = with_flow ? kNumClasses + 2 : kNumClasses;
  for (int lv = 0; lv < levels; ++lv) {
    const int n = p.pool_2x2 ? 2 : p.spp_n[lv];
    const int hs = (p.H + n - 1) / n, ws = (p.W + n - 1) / n;
    for (int cell = warp; cell < n * n; cell += 8) {
      int y0, x0, ch, cw;                                // cell origin and the window that is averaged
      float inv;
      if (p.pool_2x2) {
        const int hh = p.H / 2, hw2 = p.W / 2;
        y0 = (cell >> 1) ? hh : 0; x0 = (cell & 1) ? hw2 : 0;
        ch = (cell >> 1) ? p.H - hh : hh; cw = (cell & 1) ? p.W - hw2 : hw2;
        inv = 1.0f / (float)(ch * cw);
      } else {
        y0 = (cell / n) * hs; x0 = (cell % n) * ws; ch = hs; cw = hs;
        inv = 1.0f / (float)(hs * hs);
      }
      if (lane < kNumClasses) s_hist[warp][lane] = 0;
      __syncwarp();
      float sx = 0.f, sy = 0.f;
      for (int i = lane; i < ch * cw; i += 32) {
        const int y = y0 + i / cw, x = x0 + i % cw;
        if (y < p.H && x < p.W) {                       // beyond the map: tf.pad zeros (an all-zero one-hot row)
          const int lab = label_at(p, seg_off, y * p.W + x);
          if (lab >= 0 && lab < kNumClasses) atomicAdd(&s_hist[warp][lab], 1);
          if (with_flow) {                              // the target's flow is zeros (davo.py:979): SE input se_in(0)
            const float2 v = f == 1 ? make_float2(0.f, 0.f) : flow1_at(p, b, f == 2 ? 1 : 0, y * p.W + x, hw);
            sx += se_in_x(v.x, p);
            sy += se_in_y(v.y, p);
          }
        }
      }
      if (with_flow) {
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) {
          sx += __shfl_xor_sync(0xffffffffu, sx, o);
          sy += __shfl_xor_sync(0xffffffffu, sy, o);
        }
      }
      __syncwarp();
      if (lane < kNumClasses) s_pool[(cell0 + cell) * cs + lane] = (float)s_hist[warp][lane] * inv;
      if (with_flow && lane == 0) {
        s_pool[(cell0 + cell) * cs + kNumClasses] = sx * inv;
        s_pool[(cell0 + cell) * cs + kNumClasses + 1] = sy * inv;
      }
      __syncwarp();
    }
    cell0 += n * n;
  }
  __syncthreads();
  se_dense_layers(p, s_pool, s_fc1, cell0 * cs, pl, fr);
}

__device__ __forceinline__ float img_norm(uint8_t v) {
  return (float)v * (1.0f / 255.0f) * 2.0f - 1.0f;     // davo.py:1519-1522
}

// Attention value of one pixel of one frame (davo.py:1115-1400 after the pooling and the dense layers).
//   w      the frame's slot of att_w: 19 class weights, or the excitation of a per-pixel source
//   w_far  depth_split only: the "far" table (the frame's slot holds the "near" one)
//   lab    the pixel's label (tf.cast(seg, int32)); r, g, b its [-1, 1] colour; d_self / d_tgt the depth of this
//          frame and of the target at the pixel; sfx, sfy the SE flow (se_in_x / se_in_y; se_in(0) on the target)
// Class-weight sources: w[lab], 0 outside 0..18 (tf.one_hot gives an all-zero row).  Per-pixel sources
// (pixel_map): reduce_sum(SE input * excitation) (attention_module.py:51; davo.py:1161, 1230, 1295, 1377).
__device__ __forceinline__ float frame_attention(const FrontParams& p, const float* w, const float* w_far, int lab,
                                                 float r, float g, float b, float d_self, float d_tgt, float sfx,
                                                 float sfy) {
  const bool in = lab >= 0 && lab < kNumClasses;
  if (p.pixel_map) {
    if (p.att_src == 4) return r * w[0] + g * w[1] + b * w[2];            // se_block(image)
    if (p.att_src == 5) {                                                 // se_block(depth term [, SE flow]); see se_pool_kernel
      const float x = p.depth_norm == 2 ? 1.0f / d_self : p.depth_norm == 1 ? (d_self + d_tgt) / 80.0f : d_self + d_tgt;
      float a = x * w[0];
      if (p.pixel_map == 2) a += sfx * w[1] + sfy * w[2];
      return a;
    }
    return (in ? w[lab] : 0.0f) + sfx * w[kNumClasses] + sfy * w[kNumClasses + 1];   // se_block(concat(one_hot, SE flow))
  }
  if (p.depth_split) return in ? (d_self < p.depth_thres ? w[lab] : w_far[lab]) : 0.0f;   // davo.py:1143-1152
  return in ? w[lab] : 0.0f;
}

// grid (kPackBlocksPerPair, npairs), 256 threads, one thread per pixel.  Writes the
// 16-channel packed pixel (davo.py:1439-1442, posenn.py:198):
//   ch 0-2  tgt r g b        ch 3-4  tgt flow (zeros)     ch 5-7  src r g b (x A)
//   ch 8-9  src flow (x A)   ch 10-12 / 13-15: the TF32 rounding residuals of ch 0-2 / 5-7.
// Every value is stored TF32-rounded (the tensor core drops the low 13 bits).  The image
// channels take only 256 x |classes| distinct values, so their rounding error would be the
// same for every pixel and sample; the residual channels (which cnv1 multiplies by the same
// weights) give them ~21 mantissa bits at no cost: the slab is 16 channels wide anyway.
// The four float4 of a pixel are transposed across each lane quad with shuffles so that
// every store instruction writes whole 64-B runs.
__device__ __forceinline__ float4 shfl_xor4(const float4 v, int m) {
  return make_float4(__shfl_xor_sync(0xffffffffu, v.x, m), __shfl_xor_sync(0xffffffffu, v.y, m),
                     __shfl_xor_sync(0xffffffffu, v.z, m), __shfl_xor_sync(0xffffffffu, v.w, m));
}

__global__ void __launch_bounds__(256) pack_kernel(const FrontParams p) {
  pdl_launch_dependents();
  pdl_wait();                     // workspace buffers are shared with the kernels before this one
  __shared__ float s_w[kAttStride], s_wt[kAttStride];      // class weights (or excitation): source frame, target frame
  const int pl = blockIdx.y;
  int b, k;
  pair_of_slot(p.pair_mode, p.pair0 + pl, &b, &k);
  const int hw = p.H * p.W;
  if (threadIdx.x < kAttStride) {
    const bool se = p.att_src == 1 || p.att_src >= 3;
    const float st = threadIdx.x < kNumClasses ? p.static_w[threadIdx.x] : 0.0f;
    s_w[threadIdx.x] = se ? p.att_w[((size_t)pl * kAttFrames + 0) * kAttStride + threadIdx.x]
                     : p.att_src == 2 ? st : 1.0f;
    s_wt[threadIdx.x] = (se && (!p.att_tgt_ones || p.depth_split)) ? p.att_w[((size_t)pl * kAttFrames + 1) * kAttStride + threadIdx.x]
                      : p.att_src == 2 ? st : 1.0f;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, j = lane & 3;
  const uint8_t* img_t = frame_img(p.in, b, 1);                // tgt = centre frame
  const uint8_t* img_s = frame_img(p.in, b, k == 0 ? 0 : 2);
  const size_t seg_src = frame_plane(p.in, b, k == 0 ? 0 : 2, hw), seg_tgt = frame_plane(p.in, b, 1, hw);
  float4* out = reinterpret_cast<float4*>(p.packed + (size_t)pl * hw * kPackedC);
  for (int base = blockIdx.x * 256; base < hw; base += kPackBlocksPerPair * 256) {
    const int pix_raw = base + threadIdx.x;
    const int pix = min(pix_raw, hw - 1);                       // keep every lane in the shuffles
    const int h = pix / p.W;                                    // (a float reciprocal picks the wrong row at some widths)
    const size_t px_off = (size_t)h * p.in.img_row + (pix - h * p.W) * 3;
    const uint8_t* pt = img_t + px_off;
    const uint8_t* ps = img_s + px_off;
    const float tr0 = img_norm(pt[0]), tg0 = img_norm(pt[1]), tb0 = img_norm(pt[2]);
    const float sr0 = img_norm(ps[0]), sg0 = img_norm(ps[1]), sb0 = img_norm(ps[2]);
    float2 fl = make_float2(0.f, 0.f);
    if (p.in_mode == 1 || (p.pixel_map && p.att_src == 6) || p.pixel_map == 2) fl = flow1_at(p, b, k, pix, hw);
    float a_src = 1.0f, a_tgt = 1.0f;
    if (p.att_src != 0) {
      const bool need_lab = !p.pixel_map || p.att_src == 6;
      const bool need_depth = p.depth_split || (p.pixel_map && p.att_src == 5);
      float ds = 0.f, dt = 0.f;
      if (need_depth) {
        dt = __ldg(p.in.depth + seg_tgt + pix);                // depth planes are placed as label planes
        ds = __ldg(p.in.depth + seg_src + pix);
      }
      const int ls = need_lab ? label_at(p, seg_src, pix) : -1;          // tf.cast truncates toward zero
      a_src = frame_attention(p, s_w, s_wt, ls, sr0, sg0, sb0, ds, dt, se_in_x(fl.x, p), se_in_y(fl.y, p));
      if (!p.att_tgt_ones) {                                             // the target's flow is zeros (davo.py:979)
        const int lt = need_lab ? label_at(p, seg_tgt, pix) : -1;
        a_tgt = frame_attention(p, s_wt, s_wt, lt, tr0, tg0, tb0, dt, dt, se_in_x(0.f, p), se_in_y(0.f, p));
      }
    }
    const float mt = p.mask_rgb ? a_tgt : 1.0f, ms = p.mask_rgb ? a_src : 1.0f;
    const float tr = tr0 * mt, tg = tg0 * mt, tb = tb0 * mt;
    const float sr = sr0 * ms, sg = sg0 * ms, sb = sb0 * ms;
    float fx = 0.f, fy = 0.f;
    if (p.in_mode == 1) {
      const float m = p.mask_flow ? a_src : 1.0f;
      fx = fl.x * m;
      fy = fl.y * m;
    }
    const float trh = round_tf32(tr), tgh = round_tf32(tg), tbh = round_tf32(tb);
    const float srh = round_tf32(sr), sgh = round_tf32(sg), sbh = round_tf32(sb);

    float4 q0 = make_float4(trh, tgh, tbh, 0.f);
    float4 q1 = make_float4(0.f, srh, sgh, sbh);
    float4 q2 = make_float4(round_tf32(fx), round_tf32(fy), round_tf32(tr - trh), round_tf32(tg - tgh));
    float4 q3 = make_float4(round_tf32(tb - tbh), round_tf32(sr - srh), round_tf32(sg - sgh),
                            round_tf32(sb - sbh));
    // 4x4 transpose across the lane quad: afterwards lane j holds quarter j of pixels 4i..4i+3
    {
      const bool up = (j & 2) != 0;                              // exchange with lane ^ 2
      const float4 s0 = shfl_xor4(up ? q0 : q2, 2), s1 = shfl_xor4(up ? q1 : q3, 2);
      if (up) { q0 = s0; q1 = s1; } else { q2 = s0; q3 = s1; }
      // now lanes 0,1 hold rows (q0,q1) of pixels {own, own^2}; lanes 2,3 hold rows (q2,q3)
      float4 a0 = up ? q2 : q0, a1 = up ? q3 : q1;               // own pixel, rows (2j'..)
      float4 b0 = up ? q0 : q2, b1 = up ? q1 : q3;               // pixel ^2
      const bool odd = (j & 1) != 0;                             // exchange with lane ^ 1
      const float4 t0 = shfl_xor4(odd ? a0 : a1, 1), t1 = shfl_xor4(odd ? b0 : b1, 1);
      if (odd) { a0 = t0; b0 = t1; } else { a1 = t0; b1 = t1; }
      // lane j now holds quarter j of: (a0: pixel j&~1 | .., a1: .. | 1, b0, b1: the ^2 pair)
      const int quad = pix_raw & ~3;
      const int pA = quad + (up ? 2 : 0), pB = quad + (up ? 0 : 2);
      if (pA + 0 < hw) out[(size_t)(pA + 0) * 4 + j] = a0;
      if (pA + 1 < hw) out[(size_t)(pA + 1) * 4 + j] = a1;
      if (pB + 0 < hw) out[(size_t)(pB + 0) * 4 + j] = b0;
      if (pB + 1 < hw) out[(size_t)(pB + 1) * 4 + j] = b1;
    }
  }
}

// 8-channel packed layout (FrontParams::packed_c == 8; W % 16 == 0): [tgt r g b, src r g b (x A),
// src flow x y (x A)], every value TF32-rounded.  grid (kPack8Blocks or a quarter of it, npairs), 256 threads, one
// thread per 4 consecutive pixels of a row: the 12 image bytes of a frame are three 32-bit
// loads, labels and flow are float4 loads.  A thread's 8 float4 (128 B) go through a per-warp
// XOR-swizzled staging buffer so that every store instruction of the warp writes 512
// consecutive bytes.
constexpr int kPack8Blocks = 52;
__device__ __forceinline__ void unpack_rgb4(uint32_t t0, uint32_t t1, uint32_t t2, float (&r)[4], float (&g)[4],
                                            float (&b)[4]) {
  r[0] = img_norm(t0 & 255u); g[0] = img_norm((t0 >> 8) & 255u); b[0] = img_norm((t0 >> 16) & 255u);
  r[1] = img_norm(t0 >> 24); g[1] = img_norm(t1 & 255u); b[1] = img_norm((t1 >> 8) & 255u);
  r[2] = img_norm((t1 >> 16) & 255u); g[2] = img_norm(t1 >> 24); b[2] = img_norm(t2 & 255u);
  r[3] = img_norm((t2 >> 8) & 255u); g[3] = img_norm((t2 >> 16) & 255u); b[3] = img_norm(t2 >> 24);
}

// One 128-B slab of the 8-channel packed layout: 4 consecutive pixels x [tgt r g b, src r g b (x A), src flow x y (x A)],
// every value TF32-rounded.  t0..t2 / s0..s2: the 12 image bytes of the target / source frame; ls / lt: labels as
// tf.cast gives them (anything outside 0..18: no class); f0, f1: the flow of pixels (0, 1) and (2, 3).  s_w / s_wt: the
// class weights of the source / target frame.  Shared by pack8_kernel and the fused front end of cnv1 (conv_pm.cuh), so
// that both produce the same bits.
__device__ __forceinline__ void pack8_quad(const FrontParams& p, const float* s_w, const float* s_wt, uint32_t t0, uint32_t t1,
                                           uint32_t t2, uint32_t s0, uint32_t s1, uint32_t s2, const int (&ls)[4], const int (&lt)[4],
                                           const float4 f0, const float4 f1, float4 (&q)[8]) {
  float tr[4], tg[4], tb[4], sr[4], sg[4], sb[4], a_src[4] = {1.f, 1.f, 1.f, 1.f}, a_tgt[4] = {1.f, 1.f, 1.f, 1.f};
  unpack_rgb4(t0, t1, t2, tr, tg, tb);
  unpack_rgb4(s0, s1, s2, sr, sg, sb);
  if (p.att_src != 0) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
      a_src[i] = (ls[i] >= 0 && ls[i] < kNumClasses) ? s_w[ls[i]] : 0.0f;   // one_hot: out of range -> 0
    if (!p.att_tgt_ones) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        a_tgt[i] = (lt[i] >= 0 && lt[i] < kNumClasses) ? s_wt[lt[i]] : 0.0f;
    }
  }
  float fx[4] = {0.f, 0.f, 0.f, 0.f}, fy[4] = {0.f, 0.f, 0.f, 0.f};
  if (p.in_mode == 1) {
    fx[0] = f0.x; fy[0] = f0.y; fx[1] = f0.z; fy[1] = f0.w;
    fx[2] = f1.x; fy[2] = f1.y; fx[3] = f1.z; fy[3] = f1.w;
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float mt = p.mask_rgb ? a_tgt[i] : 1.0f, ms = p.mask_rgb ? a_src[i] : 1.0f;
    const float mf = p.mask_flow ? a_src[i] : 1.0f;
    // image values are finite (bytes times class weights): the two-instruction form of the rounding, bit-equal to
    // cvt.rna.tf32 on every finite float32 (tools/experiments/tf32_round.cu: all 2^32 patterns); the flow keeps cvt.rna
    q[2 * i + 0] = make_float4(round_tf32_finite(tr[i] * mt), round_tf32_finite(tg[i] * mt), round_tf32_finite(tb[i] * mt),
                               round_tf32_finite(sr[i] * ms));
    q[2 * i + 1] = make_float4(round_tf32_finite(sg[i] * ms), round_tf32_finite(sb[i] * ms), round_tf32(fx[i] * mf),
                               round_tf32(fy[i] * mf));
  }
}

// The body of pack8_kernel for block bx of nbx of unit pl.  Also called by front_pipeline_kernel.
__device__ __forceinline__ void pack8_body(const FrontParams& p, const int bx, const int nbx, const int pl) {
  __shared__ float s_w[kNumClasses], s_wt[kNumClasses];    // class weights: source frame, target frame
  __shared__ float4 s_stage[8][256];
  int b, k;
  pair_of_slot(p.pair_mode, p.pair0 + pl, &b, &k);
  const int hw = p.H * p.W, groups = hw / 4;
  if (threadIdx.x < kNumClasses) {
    const bool se = p.att_src == 1 || p.att_src >= 3;
    s_w[threadIdx.x] = se ? __ldcg(p.att_w + ((size_t)pl * kAttFrames + 0) * kAttStride + threadIdx.x)
                     : p.att_src == 2 ? p.static_w[threadIdx.x] : 1.0f;
    s_wt[threadIdx.x] = (se && !p.att_tgt_ones) ? __ldcg(p.att_w + ((size_t)pl * kAttFrames + 1) * kAttStride + threadIdx.x)
                      : p.att_src == 2 ? p.static_w[threadIdx.x] : 1.0f;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint8_t* img_t = frame_img(p.in, b, 1);
  const long long img_ds = k == 0 ? -p.in.img_frame : p.in.img_frame;   // the source frame, relative to the target
  const size_t seg_src = frame_plane(p.in, b, k == 0 ? 0 : 2, hw), seg_tgt = frame_plane(p.in, b, 1, hw);
  float4* out = reinterpret_cast<float4*>(p.packed + (size_t)pl * hw * 8);
  float4* st = s_stage[warp];
  for (int base = bx * 256; base < groups; base += nbx * 256) {
    const int gi = base + threadIdx.x;
    float4 q[8];
    if (gi < groups) {
      const int p0 = gi * 4, h = p0 / p.W, w = p0 - h * p.W;
      const size_t px_off = (size_t)h * p.in.img_row + w * 3;
      const uint32_t* pt = reinterpret_cast<const uint32_t*>(img_t + px_off);
      const uint32_t* ps = reinterpret_cast<const uint32_t*>(img_t + img_ds + px_off);
      int lsv[4] = {-1, -1, -1, -1}, ltv[4] = {-1, -1, -1, -1};
      if (p.att_src != 0) {
        labels4_at(p, seg_src, p0, lsv);                            // tf.cast truncates toward zero
        if (!p.att_tgt_ones) labels4_at(p, seg_tgt, p0, ltv);
      }
      float4 f0 = make_float4(0.f, 0.f, 0.f, 0.f), f1 = f0;
      if (p.in_mode == 1) { f0 = flow2_at(p, b, k, p0, hw); f1 = flow2_at(p, b, k, p0 + 2, hw); }
      pack8_quad(p, s_w, s_wt, __ldg(pt), __ldg(pt + 1), __ldg(pt + 2), __ldg(ps), __ldg(ps + 1), __ldg(ps + 2), lsv, ltv, f0, f1, q);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) st[8 * lane + (j ^ (lane & 7))] = q[j];
    __syncwarp();
    const size_t f4_0 = (size_t)(base + warp * 32) * 8;          // first float4 of this warp's 32 groups
#pragma unroll
    for (int J = 0; J < 8; ++J) {
      const int i = J * 32 + lane, Lp = i >> 3, jp = i & 7;
      const float4 v = st[8 * Lp + (jp ^ (Lp & 7))];
      if (f4_0 + i < (size_t)hw * 2) out[f4_0 + i] = v;
    }
    __syncwarp();
  }
}

__global__ void __launch_bounds__(256, 4) pack8_kernel(const FrontParams p) {
  pdl_launch_dependents();
  pdl_wait();                     // workspace buffers are shared with the kernels before this one
  pack8_body(p, blockIdx.x, gridDim.x, blockIdx.y);
}

// ---- the whole front end of a pass in ONE launch (se_flow with global pooling, 8-channel packed layout) ----
// Persistent blocks take work items from a global counter, in order.  Step t of the schedule holds the 16 pooling
// items of frame pair t and the kPipePack packing items of frame pair t - kPipeLook: a pair is packed a few steps after it
// was pooled, so the second read of its flow planes comes out of L2 instead of HBM, and the latency-bound pooling runs
// next to the streaming pack instead of in front of it.  A packing item waits for its pair's class weights (a flag the
// pooling block that finished the pair sets); every item it can wait for has a smaller index and was therefore already
// taken by a running block that never waits: no deadlock.  The arithmetic of every item is the separate kernels', so
// the results are the same bits.
constexpr int kPipePack = 13;        // packing items per pair (as pack8_kernel's grid on full passes)
constexpr int kPipeLook = 4;         // pairs pooled ahead of the pair being packed (1.7 MB of flow: L2-resident)
struct FrontPipe {
  int* next;                         // work counter, zero between launches
  int* done;                         // blocks that have left, zero between launches
  unsigned int* launches;            // completed launches: kept on the DEVICE so that a replayed CUDA graph (whose kernel
                                     // arguments are frozen) still sees a new number every time
  unsigned int* ready;               // [mb] number of the launch in which the pair's class weights were written
};

__global__ void __launch_bounds__(256, 4) front_pipeline_kernel(const FrontParams p, const FrontPipe q) {
  pdl_launch_dependents();
  pdl_wait();                     // workspace buffers are shared with the kernels before this one
  __shared__ int s_item;
  // this launch's number: the counter moves only when the LAST block of a launch leaves, i.e. after every block of that
  // launch (this one included) has read it
  const unsigned int epoch = *reinterpret_cast<volatile unsigned int*>(q.launches) + 1u;
  constexpr int kStep = kPoolSplits + kPipePack;
  const int total = (p.npairs + kPipeLook) * kStep;
  for (;;) {
    __syncthreads();                                     // everyone is done with the previous item (and with s_item)
    if (threadIdx.x == 0) s_item = atomicAdd(q.next, 1);
    __syncthreads();
    const int item = s_item;
    if (item >= total) break;
    const int t = item / kStep, j = item - t * kStep;
    if (j < kPoolSplits) {
      if (t < p.npairs) {
        const bool finished = se_pool_body(p, j, t, 0);
        if (finished) {                                  // block-uniform
          __syncthreads();                               // the class weights of every thread are written ...
          if (threadIdx.x == 0) { __threadfence(); atomicExch(&q.ready[t], epoch); }   // ... and visible before the flag
        }
      }
    } else {
      const int pl = t - kPipeLook;
      if (pl >= 0) {
        if (threadIdx.x == 0) {
          const long long t0 = clock64();                   // bounded like every other wait: a protocol bug traps, never hangs
          while (atomicAdd(&q.ready[pl], 0u) != epoch) {
            __nanosleep(100);
            if (clock64() - t0 > 4000000000LL) __trap();
          }
          __threadfence();
        }
        __syncthreads();
        pack8_body(p, j - kPoolSplits, kPipePack, pl);
      }
    }
  }
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(q.done, 1) == (int)gridDim.x - 1) {      // the last block leaves the counters ready for the next launch
      *q.next = 0; *q.done = 0; *q.launches = epoch;
      __threadfence();
    }
  }
}

// Sample units (non-shared nets, posenn.py:12-131: inputs = concat(tgt, src0, src1)): 16 packed
// channels per pixel:  0-2 tgt rgb (x A_tgt), 3-5 src0 rgb, 6-7 src0 flow (x A_0),
// 8-10 src1 rgb, 11-12 src1 flow (x A_1), 13-15 zero.  grid (kPackBlocksPerPair, units), one
// thread per pixel.
__global__ void __launch_bounds__(256) pack_sample_kernel(const FrontParams p) {
  pdl_launch_dependents();
  pdl_wait();                     // workspace buffers are shared with the kernels before this one
  // class weights (or excitation) of slots src0, src1, tgt; with the depth-split source (target map = ones) the four
  // slots are src0 near, src0 far, src1 near, src1 far
  __shared__ float s_w[kAttFrames][kAttStride];
  const int pl = blockIdx.y;
  int b, k;
  pair_of_slot(p.pair_mode, p.pair0 + pl, &b, &k);
  const int hw = p.H * p.W;
  for (int t = threadIdx.x; t < kAttFrames * kAttStride; t += blockDim.x) {
    const int fr = t / kAttStride, c = t % kAttStride;
    const bool se = p.att_src == 1 || p.att_src >= 3;
    float v = 1.0f;
    if (p.att_src == 2) v = c < kNumClasses ? p.static_w[c] : 0.0f;
    else if (se && (p.depth_split || (fr < 3 && !(fr == 2 && p.att_tgt_ones)))) v = p.att_w[((size_t)pl * kAttFrames + fr) * kAttStride + c];
    s_w[fr][c] = v;
  }
  __syncthreads();
  const bool need_lab = !p.pixel_map || p.att_src == 6;
  const bool need_depth = p.depth_split || (p.pixel_map && p.att_src == 5);
  const bool need_seflow = (p.pixel_map && p.att_src == 6) || p.pixel_map == 2;
  float4* out = reinterpret_cast<float4*>(p.packed + (size_t)pl * hw * 16);
  for (int pix = blockIdx.x * 256 + threadIdx.x; pix < hw; pix += kPackBlocksPerPair * 256) {
    const int h = pix / p.W, w = pix - h * p.W;
    const size_t px_off = (size_t)h * p.in.img_row + w * 3;
    float a[3] = {1.f, 1.f, 1.f};                            // A_src0, A_src1, A_tgt
    if (p.att_src != 0) {
      const float dt = need_depth ? __ldg(p.in.depth + frame_plane(p.in, b, 1, hw) + pix) : 0.f;
#pragma unroll
      for (int fr = 0; fr < 3; ++fr) {
        if (fr == 2 && p.att_tgt_ones) continue;
        const int plane = unit_frame(1, 0, fr);              // 0 = src0, 2 = src1, 1 = tgt: label / depth plane, image column block
        const int lab = need_lab ? label_at(p, frame_plane(p.in, b, plane, hw), pix) : -1;   // tf.cast truncates
        float r = 0.f, g = 0.f, bl = 0.f, ds = 0.f, sfx = se_in_x(0.f, p), sfy = se_in_y(0.f, p);   // the target's flow is zeros (davo.py:979)
        if (p.pixel_map && p.att_src == 4) {
          const uint8_t* pf = frame_img(p.in, b, plane) + px_off;
          r = img_norm(pf[0]); g = img_norm(pf[1]); bl = img_norm(pf[2]);
        }
        if (need_depth) ds = __ldg(p.in.depth + frame_plane(p.in, b, plane, hw) + pix);
        if (need_seflow && fr != 2) {
          const float2 f = flow1_at(p, b, fr, pix, hw);      // slot 0 = src0 -> flow[:, 0], slot 1 = src1 -> flow[:, 1]
          sfx = se_in_x(f.x, p); sfy = se_in_y(f.y, p);
        }
        const float* wn = p.depth_split ? s_w[2 * fr] : s_w[fr];                       // depth_split: fr is 0 or 1 (target map = ones)
        const float* wf = p.depth_split ? s_w[2 * fr + 1] : s_w[fr];
        a[fr] = frame_attention(p, wn, wf, lab, r, g, bl, ds, dt, sfx, sfy);             // one_hot: out of range -> 0
      }
    }
    float v[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = 0.f;
    const float mt = p.mask_rgb ? a[2] : 1.0f;
    const uint8_t* pt = frame_img(p.in, b, 1) + px_off;
#pragma unroll
    for (int c = 0; c < 3; ++c) v[c] = img_norm(pt[c]) * mt;
#pragma unroll
    for (int sidx = 0; sidx < 2; ++sidx) {
      const float ms = p.mask_rgb ? a[sidx] : 1.0f, mf = p.mask_flow ? a[sidx] : 1.0f;
      const uint8_t* ps = frame_img(p.in, b, sidx == 0 ? 0 : 2) + px_off;
#pragma unroll
      for (int c = 0; c < 3; ++c) v[3 + 5 * sidx + c] = img_norm(ps[c]) * ms;
      if (p.in_mode == 1) {
        const float2 f = flow1_at(p, b, sidx, pix, hw);
        v[6 + 5 * sidx] = f.x * mf;
        v[7 + 5 * sidx] = f.y * mf;
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q)
      out[(size_t)pix * 4 + q] = make_float4(round_tf32(v[4 * q]), round_tf32(v[4 * q + 1]), round_tf32(v[4 * q + 2]),
                                             round_tf32(v[4 * q + 3]));
  }
}

struct HeadParams {
  int pair0, npairs, pair_mode;
  int nbr;                // branches: 2 (rotation, translation) or 1 (couple nets)
  int nsrc;               // source frames per unit: 1 (shared nets: a frame pair) or 2 (a whole sample)
  int nparts;             // partial rows per (pair, branch) = tiles * 4
  float inv_hw;           // 1 / (H7 * W7)
  const float* sums;      // [mb][nbr][nparts][256]
  const float* wpred;     // [nbr][256][per], per = 6 * nsrc / nbr outputs of a branch's pred conv
  const float* bpred;     // [nbr][per]
  float* pose_out;        // [B][2][6]
};

// grid units, 256 threads.  mean_{h,w} pred(cnv7) == pred(mean_{h,w} cnv7): pred is linear
// (posenn.py:240-241); pose = 0.01 * [rot(3), trans(3)] per source frame:
//   decouple nets: branch avg [3*nsrc] -> [nsrc, 3], rot | trans concatenated (posenn.py:121-123, 248-250)
//   couple nets:   avg [6*nsrc] -> [nsrc, 6]                                     (posenn.py:62, 183)
__global__ void __launch_bounds__(256) head_kernel(const HeadParams p) {
  pdl_launch_dependents();
  pdl_wait();                     // workspace buffers are shared with the kernels before this one
  __shared__ float s_mean[2][256];
  const int pl = blockIdx.x;
  const int c = threadIdx.x;
  for (int br = 0; br < p.nbr; ++br) {
    const float* src = p.sums + ((size_t)(pl * p.nbr + br) * p.nparts) * 256 + c;
    float a = 0.f;
    for (int i = 0; i < p.nparts; ++i) a += src[(size_t)i * 256];
    s_mean[br][c] = a * p.inv_hw;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int per = 6 * p.nsrc / p.nbr;            // outputs per branch
  int b, k;
  pair_of_slot(p.pair_mode, p.pair0 + pl, &b, &k);
  for (int o = warp; o < 6 * p.nsrc; o += 8) {
    const int br = o / per, j = o % per;
    float a = 0.f;
    for (int i = lane; i < 256; i += 32) a += s_mean[br][i] * p.wpred[(br * 256 + i) * per + j];
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) a += __shfl_xor_sync(0xffffffffu, a, off);
    if (lane == 0) {
      // where output j of branch br lands in pose[b][source][6]
      const int comps = 6 / p.nbr;               // components a branch contributes per source: 3 or 6
      const int src = p.nsrc == 1 ? k : j / comps, comp = br * comps + j % comps;
      p.pose_out[(size_t)(b * 2 + src) * 6 + comp] = 0.01f * (a + p.bpred[br * per + j]);
    }
  }
}

// ------------------------------------------------------------------------------
// `-se_insert` (reference nets/posenn.py:225-228): se_block(cnv5, 'cnv5_se_attention', ratio=8)
// in front of cnv6 of each branch.  cnv5 is RE-ASSIGNED inside the branch loop, so the
// translation branch's block sits on top of the rotation branch's output:
//     exc_r = SE_r(mean cnv5),  cnv6_rot   = conv(cnv5 * exc_r)
//     exc_t = SE_t(mean(cnv5 * exc_r)) = SE_t(mean(cnv5) * exc_r),  cnv6_trans = conv(cnv5 * exc_r * exc_t)
// The excitation is per channel, so the second block needs no second pass over the map.
constexpr int kSe5Splits = 32;
struct Se5Params {
  int npairs, hw;               // pixels of the cnv5 map as stored (with its pitch; pad pixels are zeros)
  float inv_n;                  // 1 / (pixels of the map proper): the divisor of the global average pool
  int nbr;                      // branches (2: rotation then translation; 1: couple nets)
  int stack;                    // 1: -se_insert, where cnv5 is RE-ASSIGNED in the branch loop (posenn.py:227), so the
                                //    second branch's block sees and scales the first one's output;
                                // 0: -se_replace (posenn.py:234-236): every branch excites the original cnv5
  int skipadd;                  // 1: -se_skipadd (posenn.py:229-233): the block sits on cnv6 (256 channels per branch,
                                //    `cnv6` below) and the result is relu(cnv5 + cnv6 * excitation)
  const float* cnv5;            // [mb][hw][256]
  const float* cnv6;            // skipadd: [mb][hw][nbr*256]
  const float* w;               // per branch: W1[256][32] b1[32] W2[32][256] b2[256]
  float* part;                  // [mb][kSe5Splits][256] (skipadd: [mb][kSe5Splits][nbr][256])
  unsigned int* count;          // [mb]
  float* scale;                 // [mb][nbr][256]: exc_r, exc_r * exc_t (stack) or exc_r, exc_t
  float* out;                   // [mb][hw][nbr*256]: cnv5 * scale[0] | cnv5 * scale[1], TF32-rounded
                                //   (skipadd: relu(cnv5 + cnv6[br] * scale[br]))
};
constexpr int kSe5BranchFloats = 256 * 32 + 32 + 32 * 256 + 256;

// grid (kSe5Splits, npairs), 256 threads (thread = channel).
__global__ void __launch_bounds__(256) se5_excite_kernel(const Se5Params p) {
  pdl_launch_dependents();
  pdl_wait();                     // workspace buffers are shared with the kernels before this one
  const int pl = blockIdx.y, c = threadIdx.x;
  const int per = (p.hw + kSe5Splits - 1) / kSe5Splits;
  const int beg = blockIdx.x * per, end = min(beg + per, p.hw);
  const int npool = p.skipadd ? p.nbr : 1;                   // pooled maps: cnv5, or every branch's cnv6
  for (int q = 0; q < npool; ++q) {
    const float* src = p.skipadd ? p.cnv6 + (size_t)pl * p.hw * (p.nbr * 256) + q * 256 + c : p.cnv5 + (size_t)pl * p.hw * 256 + c;
    const size_t stride = p.skipadd ? (size_t)p.nbr * 256 : 256;
    float a = 0.f;
    for (int i = beg; i < end; ++i) a += src[(size_t)i * stride];
    p.part[(((size_t)pl * kSe5Splits + blockIdx.x) * npool + q) * 256 + c] = a;
  }
  __shared__ int s_last;
  __shared__ float s_mean[256], s_hid[32];
  __syncthreads();
  if (c == 0) {
    __threadfence();
    const unsigned int done = atomicAdd(&p.count[pl], 1u);
    s_last = (done == kSe5Splits - 1);
    if (s_last) p.count[pl] = 0;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  float m[2] = {0.f, 0.f};
  for (int q = 0; q < npool; ++q) {
    for (int sp = 0; sp < kSe5Splits; ++sp) m[q] += __ldcg(p.part + (((size_t)pl * kSe5Splits + sp) * npool + q) * 256 + c);
    m[q] *= p.inv_n;
  }
  float scale = 1.0f;
  for (int br = 0; br < p.nbr; ++br) {
    const float* W1 = p.w + br * kSe5BranchFloats;       // [256][32]
    const float* b1 = W1 + 256 * 32;
    const float* W2 = b1 + 32;                           // [32][256]
    const float* b2 = W2 + 32 * 256;
    s_mean[c] = p.skipadd ? m[br] : m[0] * (p.stack ? scale : 1.0f);     // mean of what this branch's block sees
    __syncthreads();
    if (c < 32) {
      float h = b1[c];
      for (int i = 0; i < 256; ++i) h += s_mean[i] * W1[i * 32 + c];
      s_hid[c] = fmaxf(h, 0.f);                          // se_block's default activation: relu
    }
    __syncthreads();
    float e = b2[c];
    for (int j = 0; j < 32; ++j) e += s_hid[j] * W2[j * 256 + c];
    const float exc = 1.0f / (1.0f + expf(-e));
    scale = p.stack ? scale * exc : exc;
    p.scale[((size_t)pl * p.nbr + br) * 256 + c] = scale;
    __syncthreads();
  }
}

// one thread per (pixel, 4 channels): out[pixel][br*256 + c] = tf32(cnv5[pixel][c] * scale[br][c]);
// skipadd: tf32(relu(cnv5[pixel][c] + cnv6[pixel][br*256 + c] * scale[br][c]))
__global__ void __launch_bounds__(256) se5_scale_kernel(const Se5Params p) {
  pdl_launch_dependents();
  pdl_wait();                     // workspace buffers are shared with the kernels before this one
  const long long total = (long long)p.npairs * p.hw * 64;
  const long long idx = (long long)blockIdx.x * 256 + threadIdx.x;
  if (idx >= total) return;
  const int c4 = (int)(idx & 63);
  const long long pix = idx >> 6;                         // global pixel index over the pass
  const int pl = (int)(pix / p.hw);
  const float4 v = __ldg(reinterpret_cast<const float4*>(p.cnv5) + pix * 64 + c4);
  float4* o = reinterpret_cast<float4*>(p.out) + pix * 64 * p.nbr + c4;
  for (int br = 0; br < p.nbr; ++br) {
    const float4 sc = *reinterpret_cast<const float4*>(p.scale + ((size_t)pl * p.nbr + br) * 256 + c4 * 4);
    if (p.skipadd) {
      const float4 u = __ldg(reinterpret_cast<const float4*>(p.cnv6) + pix * 64 * p.nbr + br * 64 + c4);
      o[br * 64] = make_float4(round_tf32(fmaxf(v.x + u.x * sc.x, 0.f)), round_tf32(fmaxf(v.y + u.y * sc.y, 0.f)),
                               round_tf32(fmaxf(v.z + u.z * sc.z, 0.f)), round_tf32(fmaxf(v.w + u.w * sc.w, 0.f)));
    } else {
      o[br * 64] = make_float4(round_tf32(v.x * sc.x), round_tf32(v.y * sc.y), round_tf32(v.z * sc.z),
                               round_tf32(v.w * sc.w));
    }
  }
}

// ------------------------------------------------------------------------------
// Plain fp32 direct convolution (CUDA cores).  NOT on the product path: it is the
// on-GPU cross-check the tests use to tell a tcgen05/TMA descriptor error from a
// host-side packing error (davo_debug_set_conv_impl).
struct DirectConvParams {
  int npairs, Hin, Win, Cin_total, cin_off, Cin;   // input view + channels used
  int Hout, Wout, Cout, out_stride, cout_off;
  int kh, kw, stride, dil, pad_t, pad_l;
  int relu, round_out;
  int cmap[16];          // weight input channel -> input tensor channel (cnv1 only), else identity
  int use_cmap;
  const float* in;       // [n][Hin][Win][Cin_total]
  const float* w;        // HWIO [kh][kw][Cin][Cout]
  const float* bias;     // [Cout]
  float* out;            // [n][Hout][Wout][out_stride]
};

__global__ void __launch_bounds__(256) conv_direct_kernel(const DirectConvParams p) {
  const long long total = (long long)p.npairs * p.Hout * p.Wout * p.Cout;
  const long long idx = (long long)blockIdx.x * 256 + threadIdx.x;
  if (idx >= total) return;
  const int co = (int)(idx % p.Cout);
  long long r = idx / p.Cout;
  const int ow = (int)(r % p.Wout);
  r /= p.Wout;
  const int oh = (int)(r % p.Hout);
  const int n = (int)(r / p.Hout);
  float acc = p.bias[co];
  for (int ty = 0; ty < p.kh; ++ty) {
    const int ih = oh * p.stride + ty * p.dil - p.pad_t;
    if (ih < 0 || ih >= p.Hin) continue;
    for (int tx = 0; tx < p.kw; ++tx) {
      const int iw = ow * p.stride + tx * p.dil - p.pad_l;
      if (iw < 0 || iw >= p.Win) continue;
      const float* ip = p.in + ((size_t)(n * p.Hin + ih) * p.Win + iw) * p.Cin_total + p.cin_off;
      const float* wp = p.w + ((size_t)(ty * p.kw + tx) * p.Cin) * p.Cout + co;
      for (int ci = 0; ci < p.Cin; ++ci) {
        const int ic = p.use_cmap ? p.cmap[ci] : ci;
        if (ic < 0) continue;                    // a weight channel whose input is identically zero
        acc = fmaf(ip[ic], wp[(size_t)ci * p.Cout], acc);
      }
    }
  }
  if (p.relu) acc = fmaxf(acc, 0.f);
  if (p.round_out) acc = round_tf32(acc);
  p.out[((size_t)(n * p.Hout + oh) * p.Wout + ow) * p.out_stride + p.cout_off + co] = acc;
}

// Spatial sum of [n][H][W][C] into the head's partial layout with nparts = 1.
__global__ void __launch_bounds__(256) spatial_sum_kernel(const float* in, int hw, int C, int cstride,
                                                          int coff, float* out /*[n][256]*/) {
  const int n = blockIdx.x, c = threadIdx.x;
  if (c >= C) return;
  float a = 0.f;
  for (int i = 0; i < hw; ++i) a += in[((size_t)n * hw + i) * cstride + coff + c];
  out[(size_t)n * 256 + c] = a;
}

}  // namespace davo
