// mode='feature' outputs of DAVO.inference (davo.py:1553-1564): what the reference fetches next to
// the poses for visualisation (consumer: generate_feature_map.py:183-380).  The pose path never
// materialises these -- attention maps and masked frames exist only inside the packed PoseNN
// input -- so this mode runs three extra HBM-bound kernels after the pass:
//   feature_frames_kernel : per frame (tgt, src0, src1): the [-1,1] image (davo.py:967-971), the
//                           attention map after the target override (davo.py:1404-1412, 1467), the
//                           masked image (davo.py:1470-1474), the one-hot labels (davo.py:1115) and
//                           the Cityscapes colouring of the labels (davo.py:1005)
//   flow_maxrad_kernel + flow_color_kernel : the Middlebury colouring of the two source flows as
//                           uint8 (davo.py:988-989, utils/flow_utils.py:240-272, 461-500)
//   resize_bilinear_kernel: cnv6 of the last PoseNN call, upsampled to the input size
//                           (davo.py:1463-1465, TF 1.x resize_bilinear with align_corners=False)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "frontend.cuh"

namespace davo {

struct FeatureParams {
  FrontParams fp;         // the variant's flags and the inputs (fp.in), as the pack kernels see them (frame_attention)
  int B, H, W;
  int unit_sample, att_src, att_tgt_ones, mask_rgb;
  const float* att_w;     // [units][kAttFrames][kAttStride] of the pass that just ran (pair mode 'all')
  const float* static_w;  // [19]
  const float* wheel;     // [55][3] Middlebury colour wheel / 255 (double division, then fp32), built by the host
  // outputs, frame order f = 0 tgt, 1 src0, 2 src1 (the order of the reference's lists); any may be NULL
  float* image;           // [3][B][H][W][3]
  float* attention;       // [3][B][H][W]
  float* masked_image;    // [3][B][H][W][3]
  float* seg_19;          // [3][B][H][W][19]
  uint8_t* seg_color;     // [3][B][H][W][3]
  uint8_t* flow_color;    // [2][B][H][W][3]   src0, src1
  unsigned int* maxrad;   // [2] bit patterns of the largest flow magnitude per source (non-negative floats order as ints)
};

// Cityscapes palette, the 19 train ids (utils/seg_utils/get_dataset_colormap.py:208-234); every
// other byte value maps to black (the table there is zeros((256,3)) with these rows filled).
__constant__ uint8_t c_cityscapes[kNumClasses][3] = {
    {128, 64, 128}, {244, 35, 232}, {70, 70, 70}, {102, 102, 156}, {190, 153, 153}, {153, 153, 153},
    {250, 170, 30}, {220, 220, 0}, {107, 142, 35}, {152, 251, 152}, {70, 130, 180}, {220, 20, 60},
    {255, 0, 0}, {0, 0, 142}, {0, 0, 70}, {0, 60, 100}, {0, 80, 100}, {0, 0, 230}, {119, 11, 32}};

// Class weights of frame f of sample b, or NULL when the map is all ones (tf.ones_like: davo.py
// 1385-1389 for -no_segmask, 1408-1412 / 1218 / 1283 / 1310 / 1393 for the forced target map).
__device__ __forceinline__ const float* frame_weights(const FeatureParams& p, int b, int f) {
  if (p.att_src == 0) return nullptr;
  if (f == 0 && p.att_tgt_ones) return nullptr;
  if (p.att_src == 2) return p.static_w;
  // slots of a unit: frontend.cuh unit_frame
  if (p.unit_sample && p.fp.depth_split) return p.att_w + ((size_t)b * kAttFrames + 2 * (f - 1)) * kAttStride;   // (near, far) of src f-1
  if (p.unit_sample) return p.att_w + ((size_t)b * kAttFrames + (f == 0 ? 2 : f - 1)) * kAttStride;
  if (f == 0) return p.att_w + ((size_t)(2 * b) * kAttFrames + 1) * kAttStride;
  return p.att_w + ((size_t)(2 * b + (f - 1)) * kAttFrames + 0) * kAttStride;
}

// grid (blocks, B, 3 frames); a thread takes 4 consecutive pixels of a row
__global__ void __launch_bounds__(256) feature_frames_kernel(const FeatureParams p) {
  __shared__ float s_w[kAttStride], s_wf[kAttStride];      // the frame's table, and the "far" table of a depth-split source
  __shared__ int s_ones;
  const int b = blockIdx.y, f = blockIdx.z;
  const int hw = p.H * p.W, groups = hw / 4;
  if (threadIdx.x == 0) s_ones = frame_weights(p, b, f) == nullptr;
  if (threadIdx.x < kAttStride) {
    const float* w = frame_weights(p, b, f);
    const bool table = p.att_src != 2 || threadIdx.x < kNumClasses;        // static_w holds 19 values
    s_w[threadIdx.x] = (w && table) ? w[threadIdx.x] : 1.0f;
    s_wf[threadIdx.x] = (w && p.fp.depth_split) ? w[kAttStride + threadIdx.x] : 0.0f;   // slot 1 of the same pair
  }
  __syncthreads();
  const bool need_depth = p.fp.depth_split || (p.fp.pixel_map && p.att_src == 5);
  const bool need_flow = p.fp.pixel_map && (p.att_src == 6 || p.fp.pixel_map == 2);
  const bool ones = s_ones != 0;
  const int plane = f == 0 ? 1 : f == 1 ? 0 : 2;        // position in the inputs: [src0, tgt, src1]
  const InputView& in = p.fp.in;
  const uint8_t* img_f = frame_img(in, b, plane);
  const float* seg_p = in.seg ? in.seg + frame_plane(in, b, plane, hw) : nullptr;
  const size_t fb = (size_t)f * p.B + b;
  for (int gi = blockIdx.x * blockDim.x + threadIdx.x; gi < groups; gi += gridDim.x * blockDim.x) {
    const int p0 = gi * 4, h = p0 / p.W, w = p0 - h * p.W;
    const uint32_t* px = reinterpret_cast<const uint32_t*>(img_f + (size_t)h * in.img_row + w * 3);
    float r[4], g[4], bl[4];
    unpack_rgb4(__ldg(px), __ldg(px + 1), __ldg(px + 2), r, g, bl);
    int lab[4] = {-1, -1, -1, -1};
    if (seg_p) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(seg_p + p0));
      lab[0] = label_of(v.x); lab[1] = label_of(v.y); lab[2] = label_of(v.z); lab[3] = label_of(v.w);   // tf.cast truncates
    }
    float a[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (ones) { a[i] = 1.0f; continue; }
      float ds = 0.f, dt = 0.f, sfx = se_in_x(0.f, p.fp), sfy = se_in_y(0.f, p.fp);   // the target's flow is zeros
      if (need_depth) {
        ds = __ldg(in.depth + frame_plane(in, b, plane, hw) + p0 + i);
        dt = __ldg(in.depth + frame_plane(in, b, 1, hw) + p0 + i);
      }
      if (need_flow && f != 0) {
        const float2 v = flow1_at(p.fp, b, f - 1, p0 + i, hw);
        sfx = se_in_x(v.x, p.fp);
        sfy = se_in_y(v.y, p.fp);
      }
      a[i] = frame_attention(p.fp, s_w, s_wf, lab[i], r[i], g[i], bl[i], ds, dt, sfx, sfy);
    }
    const size_t px0 = fb * hw + p0;
    if (p.attention) *reinterpret_cast<float4*>(p.attention + px0) = make_float4(a[0], a[1], a[2], a[3]);
    if (p.image) {
      float4* o = reinterpret_cast<float4*>(p.image + px0 * 3);
      o[0] = make_float4(r[0], g[0], bl[0], r[1]);
      o[1] = make_float4(g[1], bl[1], r[2], g[2]);
      o[2] = make_float4(bl[2], r[3], g[3], bl[3]);
    }
    if (p.masked_image) {
      float m[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) m[i] = p.mask_rgb ? a[i] : 1.0f;
      float4* o = reinterpret_cast<float4*>(p.masked_image + px0 * 3);
      o[0] = make_float4(r[0] * m[0], g[0] * m[0], bl[0] * m[0], r[1] * m[1]);
      o[1] = make_float4(g[1] * m[1], bl[1] * m[1], r[2] * m[2], g[2] * m[2]);
      o[2] = make_float4(bl[2] * m[2], r[3] * m[3], g[3] * m[3], bl[3] * m[3]);
    }
    if (p.seg_19) {
      float* o = p.seg_19 + px0 * kNumClasses;              // 76 consecutive floats, 16-byte aligned
#pragma unroll
      for (int j = 0; j < kNumClasses; ++j) {
        const int e0 = 4 * j;
        float t[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int e = e0 + q, pi = e / kNumClasses, c = e - pi * kNumClasses;
          t[q] = (lab[pi] == c) ? 1.0f : 0.0f;              // one_hot: a label outside 0..18 gives a zero row
        }
        reinterpret_cast<float4*>(o)[j] = make_float4(t[0], t[1], t[2], t[3]);
      }
    }
    if (p.seg_color) {
      uint8_t c[12];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const bool in = lab[i] >= 0 && lab[i] < kNumClasses;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) c[3 * i + ch] = in ? c_cityscapes[lab[i]][ch] : (uint8_t)0;
      }
      uint32_t* o = reinterpret_cast<uint32_t*>(p.seg_color + px0 * 3);
#pragma unroll
      for (int j = 0; j < 3; ++j)
        o[j] = (uint32_t)c[4 * j] | ((uint32_t)c[4 * j + 1] << 8) | ((uint32_t)c[4 * j + 2] << 16) | ((uint32_t)c[4 * j + 3] << 24);
    }
  }
}

// ---- flow colouring ------------------------------------------------------------------------
// Every step is a separately rounded fp32 operation, as the chain of TF elementwise ops is; the
// intrinsics keep the compiler from contracting them into FMAs.
constexpr float kUnknownFlow = 1e7f;                     // utils/flow_utils.py:18
constexpr int kWheelCols = 55;                           // RY+YG+GC+CB+BM+MR = 15+6+4+11+13+6 (:551-558)

__device__ __forceinline__ float flow_rad(float u, float v) {
  return __fsqrt_rn(__fadd_rn(__fmul_rn(u, u), __fmul_rn(v, v)));
}

// grid (blocks, 2 sources): maxrad[k] = max over the WHOLE batch of |flow_k| (flow_utils.py:259-260)
__global__ void __launch_bounds__(256) flow_maxrad_kernel(const FeatureParams p) {
  const int k = blockIdx.y;
  const size_t hw = (size_t)p.H * p.W, total = (size_t)p.B * hw;
  float m = 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t b = i / hw, px = i - b * hw;
    const float2 f = __ldg(reinterpret_cast<const float2*>(flow_plane(p.fp.in, b, k) + (size_t)px * 2));
    const float u = fabsf(f.x) > kUnknownFlow ? 0.f : f.x, v = fabsf(f.y) > kUnknownFlow ? 0.f : f.y;
    m = fmaxf(m, flow_rad(u, v));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(p.maxrad + k, __float_as_uint(m));
}

__global__ void __launch_bounds__(256) flow_color_kernel(const FeatureParams p) {
  const int k = blockIdx.y;
  const size_t hw = (size_t)p.H * p.W, total = (size_t)p.B * hw;
  // maxrad = reduce_max([-1, reduce_max(rad)]); rad >= 0 so the -1 never wins
  const float denom = __fadd_rn(__uint_as_float(p.maxrad[k]), 1e-5f);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t b = i / hw, px = i - b * hw;
    const float2 f = __ldg(reinterpret_cast<const float2*>(flow_plane(p.fp.in, b, k) + (size_t)px * 2));
    float u = fabsf(f.x) > kUnknownFlow ? 0.f : f.x, v = fabsf(f.y) > kUnknownFlow ? 0.f : f.y;
    u = __fdiv_rn(u, denom);
    v = __fdiv_rn(v, denom);
    const float rad = flow_rad(u, v);
    const float a = __fdiv_rn(atan2f(-v, -u), 3.14159265358979323846f);
    const float fk = __fadd_rn(__fmul_rn(__fdiv_rn(__fadd_rn(a, 1.0f), 2.0f), (float)(kWheelCols - 1)), 1.0f);
    const float k0 = floorf(fk);
    const float fr = __fsub_rn(fk, k0);
    int idx = (int)k0 - 1;
    idx = idx < 0 ? 0 : idx >= kWheelCols ? kWheelCols - 1 : idx;
    uint8_t out[3];
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      const float c0 = __ldg(p.wheel + idx * 3 + ch);
      // flow_utils.py:490-492: col1 is assigned from col0, so the blend is (1-f)*col0 + f*col0
      float col = __fadd_rn(__fmul_rn(__fsub_rn(1.0f, fr), c0), __fmul_rn(fr, c0));
      col = rad <= 1.0f ? __fsub_rn(1.0f, __fmul_rn(rad, __fsub_rn(1.0f, col))) : __fmul_rn(col, 0.75f);
      const float img = floorf(__fmul_rn(255.0f, col));                   // :495
      // :270 img / 255, then convert_image_dtype(uint8): x * 255.5, saturate, truncate (davo.py:1530-1531)
      float s = __fmul_rn(__fdiv_rn(img, 255.0f), 255.5f);
      s = s < 0.f ? 0.f : s > 255.f ? 255.f : s;
      out[ch] = (uint8_t)s;
    }
    uint8_t* o = p.flow_color + (((size_t)k * p.B + b) * hw + px) * 3;
    o[0] = out[0]; o[1] = out[1]; o[2] = out[2];
  }
}

// ---- cnv6 upsampling -----------------------------------------------------------------------
struct ResizeParams {
  int B, H, W;            // output map
  int h, w, hp, wp;       // cnv6 map and the pitch of its buffer
  int C, cstride, coff;   // channels taken, channels per pixel of the buffer, first channel
  int unit_mul, unit_add; // unit of sample b = b * unit_mul + unit_add (the last PoseNN call: davo.py:1456-1460)
  const float* src;       // [units][hp][wp][cstride]
  float* dst;             // [B][H][W][C]
};

// tf.image.resize_bilinear, align_corners=False, TF 1.x: in = out_index * (in_size / out_size),
// lower = trunc(in), upper = min(lower + 1, in_size - 1), lerp = in - lower; rows blended after columns.
__global__ void __launch_bounds__(256) resize_bilinear_kernel(const ResizeParams p) {
  const int c4 = p.C / 4;
  const size_t total = (size_t)p.B * p.H * p.W * c4;
  const float sy = (float)p.h / (float)p.H, sx = (float)p.w / (float)p.W;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % c4);
    size_t t = i / c4;
    const int x = (int)(t % p.W); t /= p.W;
    const int y = (int)(t % p.H);
    const int b = (int)(t / p.H);
    const float fy = (float)y * sy, fx = (float)x * sx;
    const int y0 = (int)fy, x0 = (int)fx;
    const int y1 = min(y0 + 1, p.h - 1), x1 = min(x0 + 1, p.w - 1);
    const float ly = fy - (float)y0, lx = fx - (float)x0;
    const float* base = p.src + (size_t)(b * p.unit_mul + p.unit_add) * p.hp * p.wp * p.cstride + p.coff + 4 * c;
    auto at = [&](int yy, int xx) {
      return __ldg(reinterpret_cast<const float4*>(base + ((size_t)yy * p.wp + xx) * p.cstride));
    };
    const float4 tl = at(y0, x0), tr = at(y0, x1), bl = at(y1, x0), br = at(y1, x1);
    auto mix = [&](float a, float bb, float cc, float d) {
      const float top = a + (bb - a) * lx, bot = cc + (d - cc) * lx;
      return top + (bot - top) * ly;
    };
    reinterpret_cast<float4*>(p.dst)[i] = make_float4(mix(tl.x, tr.x, bl.x, br.x), mix(tl.y, tr.y, bl.y, br.y),
                                                      mix(tl.z, tr.z, bl.z, br.z), mix(tl.w, tr.w, bl.w, br.w));
  }
}

}  // namespace davo
