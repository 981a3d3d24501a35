// MXFP8 pack / unpack kernels (sm_100a): bf16 <-> [E4M3 payload | E8M0 block scales].
// Memory-bound streaming kernels: one 16-byte load (8 bf16) per thread, 4 lanes share a 32-element
// block (amax via two xor-shuffles), 8-byte payload store per thread.  Destination / source may be
// peer-mapped slab memory, so the pack can write straight across NVLink.
#include <cuda_bf16.h>
#include <cuda_fp8.h>
#include <cuda_runtime.h>

#include <cstdint>

#include "kernels/mxfp8.cuh"
#include "kernels/ptx.cuh"
#include "kernels/xfer.h"

namespace bb::gpu {
namespace {

__device__ __forceinline__ float bf16_bits_to_float(uint32_t b16) { return __uint_as_float(b16 << 16); }

__global__ void __launch_bounds__(256) mxfp8_pack_kernel(const uint4* __restrict__ src, uint64_t nblocks, uint2* __restrict__ payload,
                                                         uint8_t* __restrict__ scales) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  const uint64_t nthreads_work = nblocks * 4;  // 4 lanes per 32-element block
  for (uint64_t t = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; t < ((nthreads_work + 31) / 32) * 32; t += stride) {
    const bool active = t < nthreads_work;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (active) v = ptx::ld_nc_v4(src + t);
    float f[8];
    f[0] = bf16_bits_to_float(v.x & 0xFFFFu); f[1] = bf16_bits_to_float(v.x >> 16);
    f[2] = bf16_bits_to_float(v.y & 0xFFFFu); f[3] = bf16_bits_to_float(v.y >> 16);
    f[4] = bf16_bits_to_float(v.z & 0xFFFFu); f[5] = bf16_bits_to_float(v.z >> 16);
    f[6] = bf16_bits_to_float(v.w & 0xFFFFu); f[7] = bf16_bits_to_float(v.w >> 16);
    float amax = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float a = fabsf(f[i]);
      amax = (a > amax) ? a : amax;  // NaN compares false and is skipped
    }
    amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 1));
    amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 2));
    // shared exponent = floor(log2(amax)) - 8, stored biased (E8M0)
    int e = 127;
    if (amax > 0.f && amax < __int_as_float(0x7F800000)) {
      const int be = (__float_as_int(amax) >> 23) & 0xFF;
      e = (be == 0 ? -127 : be - 127) - 8 + 127;
      e = max(0, min(254, e));
    }
    const float inv = __int_as_float((254 - e) << 23);  // 2^(127 - e); e in [0,254] -> exponent field in [0,254]
    uint32_t lo = 0, hi = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      lo |= static_cast<uint32_t>(__nv_cvt_float_to_fp8(f[i] * inv, __NV_SATFINITE, __NV_E4M3)) << (8 * i);
      hi |= static_cast<uint32_t>(__nv_cvt_float_to_fp8(f[4 + i] * inv, __NV_SATFINITE, __NV_E4M3)) << (8 * i);
    }
    if (active) {
      payload[t] = make_uint2(lo, hi);
      if ((t & 3) == 0) scales[t >> 2] = static_cast<uint8_t>(e);
    }
  }
}

__global__ void __launch_bounds__(256) mxfp8_unpack_kernel(const uint2* __restrict__ payload, const uint8_t* __restrict__ scales,
                                                           uint64_t nblocks, uint4* __restrict__ dst) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  const uint64_t n = nblocks * 4;
  for (uint64_t t = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; t < n; t += stride) {
    const uint2 p = payload[t];
    const float s = e8m0_scale(scales[t >> 2]);
    uint32_t out[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const uint32_t w = i < 2 ? p.x : p.y;
      const uint8_t b0 = (w >> (16 * (i & 1))) & 0xFF, b1 = (w >> (16 * (i & 1) + 8)) & 0xFF;
      const float f0 = __half2float(__half(__nv_cvt_fp8_to_halfraw(b0, __NV_E4M3))) * s;
      const float f1 = __half2float(__half(__nv_cvt_fp8_to_halfraw(b1, __NV_E4M3))) * s;
      const __nv_bfloat162 h = __floats2bfloat162_rn(f0, f1);
      out[i] = *reinterpret_cast<const uint32_t*>(&h);
    }
    dst[t] = make_uint4(out[0], out[1], out[2], out[3]);
  }
}

int grid_for(uint64_t threads_needed) {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const uint64_t blocks = (threads_needed + 255) / 256;
  const uint64_t cap = static_cast<uint64_t>(sms) * 8;
  return static_cast<int>(blocks < 1 ? 1 : (blocks > cap ? cap : blocks));
}

}  // namespace

int launch_mxfp8_pack(const void* src_bf16, uint64_t n_elems, void* dst_packed, void* stream) {
  if (n_elems == 0) return 0;
  if (n_elems % 32) return static_cast<int>(cudaErrorInvalidValue);
  if ((reinterpret_cast<uintptr_t>(src_bf16) & 15) || (reinterpret_cast<uintptr_t>(dst_packed) & 7)) return static_cast<int>(cudaErrorMisalignedAddress);
  const uint64_t nblocks = n_elems / 32;
  mxfp8_pack_kernel<<<grid_for(nblocks * 4), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint4*>(src_bf16), nblocks, static_cast<uint2*>(dst_packed), static_cast<uint8_t*>(dst_packed) + n_elems);
  return static_cast<int>(cudaGetLastError());
}

int launch_mxfp8_unpack(const void* src_packed, uint64_t n_elems, void* dst_bf16, void* stream) {
  if (n_elems == 0) return 0;
  if (n_elems % 32) return static_cast<int>(cudaErrorInvalidValue);
  if ((reinterpret_cast<uintptr_t>(dst_bf16) & 15) || (reinterpret_cast<uintptr_t>(src_packed) & 7)) return static_cast<int>(cudaErrorMisalignedAddress);
  const uint64_t nblocks = n_elems / 32;
  mxfp8_unpack_kernel<<<grid_for(nblocks * 4), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint2*>(src_packed), static_cast<const uint8_t*>(src_packed) + n_elems, nblocks, static_cast<uint4*>(dst_bf16));
  return static_cast<int>(cudaGetLastError());
}

}  // namespace bb::gpu
