// MXFP8 (OCP microscaling: 32-element blocks, E8M0 shared scale, E4M3 elements) — CPU reference.
// New capability required by BASELINE.json ("optional block-scaled fp8 pack/unpack"); the
// reference has no payload transforms at all (SURVEY K12).
//
// Packed object layout for n elements (n % 32 == 0):  [ n bytes E4M3 | n/32 bytes E8M0 ]
//   amax(block)       = largest |x| over the block's finite elements (NaN elements are skipped)
//   shared_exp(block) = floor(log2(amax(block))) - 8        (8 = emax of E4M3: 448 = 1.75 * 2^8)
//                       a subnormal amax counts as 2^-127
//   E8M0 byte         = clamp(shared_exp + 127, 0, 254), so every block with amax < 2^-118 gets byte 0
//                       all-zero (or all-NaN) block -> 127 (scale 1); a block holding an Inf -> 127 as well
//   element           = sat_e4m3( x * 2^(127 - E8M0 byte) ), round-to-nearest-even (ties to the even code),
//                       saturating to +-448 (0x7E / 0xFE): an Inf element packs as +-448; the sign is kept on zero
//                       (-0 and negatives that round to zero pack as 0x80); every NaN element packs as 0x7F
// Decode: E8M0 byte e is 2^(e-127) -- byte 0 is 2^-127 (a float32 subnormal, not zero); byte 255, which pack never
// writes, is 2^128 = +Inf in float32, so its block decodes to +-Inf and its zero elements to NaN.  The element is
// E4M3 value * scale formed in float32 (exact: at most 4 significant bits, no underflow below 2^-149) and rounded to
// bf16 to nearest even.  E4M3 NaN (0x7F / 0xFF) decodes to a bf16 NaN: the CPU writes 0x7FC0, the GPU kernels 0x7FFF;
// every other result is bit-identical between the three implementations (this file, kernels/mxfp8.cu,
// kernels/xfer_mxfp8.cu), which tests/test_mxfp8_conformance.py checks exhaustively.
#pragma once
#include <cstddef>
#include <cstdint>

namespace bb::mxfp8 {

constexpr size_t kBlock = 32;
inline size_t packed_bytes(size_t n_elems) { return n_elems + n_elems / kBlock; }

uint8_t float_to_e4m3_sat(float x) noexcept;  // RNE, saturating to +-448, NaN -> 0x7F
float e4m3_to_float(uint8_t v) noexcept;
uint8_t block_scale_e8m0(float amax) noexcept;
float e8m0_to_float(uint8_t e) noexcept;

// src: n bf16 values (raw uint16), dst: packed_bytes(n).  n must be a multiple of 32.
void pack_bf16(const uint16_t* src, size_t n, uint8_t* dst) noexcept;
void unpack_bf16(const uint8_t* packed, size_t n, uint16_t* dst) noexcept;

float bf16_to_float(uint16_t v) noexcept;
uint16_t float_to_bf16(float f) noexcept;  // RNE

}  // namespace bb::mxfp8
