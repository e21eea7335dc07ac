// Saved odometry sessions (include/davo_b200.h: davo_odometry_save_many, davo_odometry_load_many): the kernels between
// the sessions' carried state and a device staging area laid out exactly as the caller's blobs.
//
//   odo_save_kernel : every blob of the call into the staging area -- its header (built on the host, checksum zero)
//                     and each session's sections, zero-padded to 16 bytes -- accumulating the blob's checksum; the
//                     last block of a blob writes the checksum into the staged header
//   odo_load_kernel : every section of every staged blob into its new session's buffers, accumulating the blob's
//                     checksum (the stored checksum word read as zero); the host compares it with the stored one
// Grid (x, blobs): block row y handles blob y, its blocks share each section.  Launches do not depend on the number of
// blobs; the host cuts a call into chunks only when the staging area would outgrow its bound.
//
// The checksum of a blob of n 8-byte little-endian words w_i is  sum_i mix(w_i + (i + 1) * 0x9E3779B97F4A7C15)
// mod 2^64, with mix the output function of splitmix64.  The sum does not depend on the order its terms are added in,
// so 64-bit atomics give the bits of a sequential host (or numpy) reference.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "odometry_many.cuh"

namespace davo {

constexpr int kOdoSections = 6;                 // davo_capi.cu: carried_state (img, seg8, seg, depth, fwd, pose)
constexpr unsigned long long kOdoGolden = 0x9E3779B97F4A7C15ull;

// One blob of a save or load call (host-built, one pinned copy per call).
struct OdoBlob {
  uint8_t* blob;                                // its place in the staging area (16-byte aligned)
  const uint8_t* header;                        // save: the header, checksum zero (in the descriptor area)
  uint8_t* sec[kOdoSections];                   // the session's buffers
  unsigned long long off[kOdoSections];         // section offsets in the blob (16-byte aligned, header first)
  unsigned long long bytes[kOdoSections];       // bytes carried; the blob holds them zero-padded to 16
  unsigned long long* sum;                      // checksum accumulator, zero at launch
  unsigned int* done;                           // save: blocks of this blob that have added their part, zero at launch
};

__host__ __device__ __forceinline__ unsigned long long odo_mix(unsigned long long z) {
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

__host__ __device__ __forceinline__ unsigned long long odo_term(unsigned long long word, unsigned long long index) {
  return odo_mix(word + (index + 1) * kOdoGolden);
}

// Thread t's part of the checksum of blob words [w0, w0 + padded / 8): bytes [0, bytes) at src (8-byte aligned), the
// rest zero.  Word `skip` (the stored checksum) counts as zero.
__device__ __forceinline__ unsigned long long odo_sum(const uint8_t* src, size_t bytes, size_t padded, size_t w0,
                                                      size_t skip, size_t t, size_t stride) {
  unsigned long long acc = 0;
  const unsigned long long* s = reinterpret_cast<const unsigned long long*>(src);
  for (size_t i = t; i < padded / 8; i += stride) {
    unsigned long long w = 0;
    if (8 * i + 8 <= bytes) {
      w = __ldg(s + i);
    } else {
      for (size_t b = 8 * i; b < bytes; ++b) w |= (unsigned long long)__ldg(src + b) << (8 * (b - 8 * i));
    }
    if (w0 + i == skip) w = 0;
    acc += odo_term(w, w0 + i);
  }
  return acc;
}

// the block's sum of `acc` in thread 0
__device__ __forceinline__ unsigned long long odo_block_sum(unsigned long long acc) {
  __shared__ unsigned long long part[32];
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) part[warp] = acc;
  __syncthreads();
  acc = 0;
  if (threadIdx.x == 0)
    for (int w = 0; w < (int)(blockDim.x + 31) / 32; ++w) acc += part[w];
  return acc;
}

__device__ __forceinline__ size_t odo_pad16(size_t b) { return (b + 15) & ~(size_t)15; }

__global__ void __launch_bounds__(256) odo_save_kernel(const OdoBlob* __restrict__ blobs, unsigned header_bytes) {
  const OdoBlob& d = blobs[blockIdx.y];
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  const size_t cw = header_bytes / 8 - 1;                // the checksum word, written last by the last block
  unsigned long long acc = odo_sum(d.header, header_bytes, header_bytes, 0, cw, t, stride);
  odo_copy(d.blob, d.header, header_bytes - 8, t, stride);
#pragma unroll 1
  for (int j = 0; j < kOdoSections; ++j) {
    const size_t bytes = d.bytes[j], padded = odo_pad16(bytes);
    if (!padded) continue;
    odo_copy(d.blob + d.off[j], d.sec[j], bytes, t, stride);
    if (t < padded - bytes) d.blob[d.off[j] + bytes + t] = 0;
    acc += odo_sum(d.sec[j], bytes, padded, d.off[j] / 8, ~(size_t)0, t, stride);
  }
  acc = odo_block_sum(acc);
  if (threadIdx.x == 0) {
    atomicAdd(d.sum, acc);
    __threadfence();                                     // the part is visible before the block counts as done
    if (atomicAdd(d.done, 1u) == gridDim.x - 1)
      *reinterpret_cast<unsigned long long*>(d.blob + 8 * cw) = atomicAdd(d.sum, 0ull);
  }
}

__global__ void __launch_bounds__(256) odo_load_kernel(const OdoBlob* __restrict__ blobs, unsigned header_bytes) {
  const OdoBlob& d = blobs[blockIdx.y];
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  unsigned long long acc = odo_sum(d.blob, header_bytes, header_bytes, 0, header_bytes / 8 - 1, t, stride);
#pragma unroll 1
  for (int j = 0; j < kOdoSections; ++j) {
    const size_t bytes = d.bytes[j], padded = odo_pad16(bytes);
    if (!padded) continue;
    odo_copy(d.sec[j], d.blob + d.off[j], bytes, t, stride);
    acc += odo_sum(d.blob + d.off[j], padded, padded, d.off[j] / 8, ~(size_t)0, t, stride);
  }
  acc = odo_block_sum(acc);
  if (threadIdx.x == 0) atomicAdd(d.sum, acc);
}

}  // namespace davo
