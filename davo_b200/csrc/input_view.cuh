// Where the inputs of a batch live: the one place that knows the two input layouts.
//
// A sample b has three frames f (0 = src0, 1 = tgt, 2 = src1) and two flow planes k (0: src0 -> tgt, 1: src1 -> tgt,
// davo.py:978-982).  Every kernel that reads an input goes through the helpers below.
//
// Triplet layout (davo_forward_pairs, the reference's feed): the frames of a sample side by side,
//   img [B][H][3W][3], seg / depth [B][3][H][W], flow [B][4][H][W][2] (planes 2 and 3 are never read).
// Sequence layout (davo_forward_sequence): sample b is frames (b, b+1, b+2) of an N-frame sequence,
//   img [N][H][W][3], seg / depth [N][H][W], flow_fwd / flow_bwd [N-1][H][W][2];
//   plane 0 of sample b is flow_fwd[b] (frame b -> b+1), plane 1 is flow_bwd[b+1] (frame b+2 -> b+1).
// Only addresses differ between the layouts: the same kernels compute the same values.
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

namespace davo {

struct InputView {
  const uint8_t* img;          // frame f of sample b starts at img + b * img_sample + f * img_frame (bytes) ...
  long long img_sample, img_frame;
  int img_row;                 // ... and its rows are img_row bytes apart
  const float* seg;            // label / depth plane f of sample b: element b * plane_sample + f * H*W
  const uint8_t* seg8;         // the same labels as bytes (255 = outside 0..18), or NULL: the host entry points
  const float* depth;          // se_depth sources only
  long long plane_sample;
  const float* flow0;          // flow plane 0 / 1 of sample b: flow0 / flow1 + b * flow_sample floats, [H][W][2]
  const float* flow1;
  long long flow_sample;
  const __half* flow16_0;      // the same two planes already in binary16 (host entry points), for samples b < n_flow16;
  const __half* flow16_1;      // the others are read from flow0 / flow1
  long long flow16_sample;
  int n_flow16;
};

// Triplet layout of H x W frames.  flow16: [B][2][H][W][2] halves for the first n16 samples.
inline InputView triplet_view(int H, int W, const uint8_t* img, const float* flow, const float* seg, const uint8_t* seg8,
                              const float* depth, const void* flow16, int n16) {
  const long long hw = (long long)H * W;
  InputView v;
  v.img = img; v.img_sample = hw * 9; v.img_frame = (long long)W * 3; v.img_row = W * 9;
  v.seg = seg; v.seg8 = seg8; v.depth = depth; v.plane_sample = 3 * hw;
  v.flow0 = flow; v.flow1 = flow ? flow + 2 * hw : nullptr; v.flow_sample = 8 * hw;
  v.flow16_0 = static_cast<const __half*>(flow16); v.flow16_1 = flow16 ? v.flow16_0 + 2 * hw : nullptr;
  v.flow16_sample = 4 * hw; v.n_flow16 = flow16 ? n16 : 0;
  return v;
}

// Sequence layout: frames start at img / seg / depth (frame 0 of sample 0); fwd[b] is plane 0 of sample b and bwd[b]
// plane 1 (the caller passes flow_bwd + 1 entry).  fwd16 / bwd16: the same for the first n16 samples, in binary16.
inline InputView sequence_view(int H, int W, const uint8_t* img, const float* fwd, const float* bwd, const float* seg,
                               const uint8_t* seg8, const float* depth, const void* fwd16, const void* bwd16, int n16) {
  const long long hw = (long long)H * W;
  InputView v;
  v.img = img; v.img_sample = hw * 3; v.img_frame = hw * 3; v.img_row = W * 3;
  v.seg = seg; v.seg8 = seg8; v.depth = depth; v.plane_sample = hw;
  v.flow0 = fwd; v.flow1 = bwd; v.flow_sample = 2 * hw;
  v.flow16_0 = static_cast<const __half*>(fwd16); v.flow16_1 = static_cast<const __half*>(bwd16);
  v.flow16_sample = 2 * hw; v.n_flow16 = (fwd16 || bwd16) ? n16 : 0;
  return v;
}

// Stacked-triplet layout (davo_odometry_push_many's staging batch): the frames of a sample one after another,
//   img [B][3][H][W][3], labels as bytes (seg8) / depth [B][3][H][W], flow [B][2][H][W][2].
inline InputView stacked_view(int H, int W, const uint8_t* img, const float* flow, const uint8_t* seg8, const float* depth) {
  const long long hw = (long long)H * W;
  InputView v;
  v.img = img; v.img_sample = hw * 9; v.img_frame = hw * 3; v.img_row = W * 3;
  v.seg = nullptr; v.seg8 = seg8; v.depth = depth; v.plane_sample = 3 * hw;
  v.flow0 = flow; v.flow1 = flow ? flow + 2 * hw : nullptr; v.flow_sample = 4 * hw;
  v.flow16_0 = nullptr; v.flow16_1 = nullptr; v.flow16_sample = 0; v.n_flow16 = 0;
  return v;
}

// first byte of row 0 of frame f of sample b; pixel (h, w) is at + h * img_row + w * 3
__device__ __forceinline__ const uint8_t* frame_img(const InputView& v, int b, int f) {
  return v.img + b * v.img_sample + f * v.img_frame;
}
// element offset of label / depth plane f of sample b
__device__ __forceinline__ size_t frame_plane(const InputView& v, int b, int f, int hw) {
  return (size_t)(b * v.plane_sample) + (size_t)f * hw;
}
// flow plane k of sample b, float32 [H][W][2]
__device__ __forceinline__ const float* flow_plane(const InputView& v, int b, int k) {
  return (k ? v.flow1 : v.flow0) + b * v.flow_sample;
}
// flow plane k of sample b < n_flow16, binary16 [H][W][2]
__device__ __forceinline__ const __half* flow16_plane(const InputView& v, int b, int k) {
  return (k ? v.flow16_1 : v.flow16_0) + b * v.flow16_sample;
}

}  // namespace davo
