// Device-side E8M0 decode shared by the stand-alone (mxfp8.cu) and fused (xfer_mxfp8.cu) unpack kernels.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace bb::gpu {

// E8M0 byte e -> 2^(e-127) as float32, as e8m0_to_float in common/mxfp8.cpp decodes it.  Bytes 1..255 are the exponent
// field itself (255 gives +Inf); byte 0 is 2^-127, the float32 subnormal 0x00400000 -- `e << 23` would give 0 and zero
// the whole block.  The product with an E4M3 value is exact only while the build does not flush subnormals (no
// --use_fast_math / -ftz=true).
__device__ __forceinline__ float e8m0_scale(uint32_t e) { return __uint_as_float(e != 0 ? e << 23 : 0x00400000u); }

}  // namespace bb::gpu
