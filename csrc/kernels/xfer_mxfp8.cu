// bb_xfer_fp8: fused MXFP8 transfer kernels (sm_100a; SURVEY K12 "fp8 pack fused into put / unpack into get").
//
//   put  (PACK)   : TMA loads a 32 KiB bf16 tile -> 8 pack warps compute the E8M0 block scales and the E4M3
//                   payload *in shared memory* -> the 16 KiB payload tile is hashed in place by tcgen05.mma
//                   (BBH64, same tile hash as bb_xfer) -> TMA stores payload + 512 B of scales to the
//                   (peer) slab -- to up to 3 replicas of the object from the one converted tile.  The bf16 data
//                   is read from HBM once and only the 0.52x packed bytes cross NVLink (once per replica).
//   get  (UNPACK) : TMA loads payload tile + scales from the slab -> tensor-core hash of the payload tile ->
//                   8 unpack warps expand to bf16 in shared memory -> TMA stores the 32 KiB tile to the caller.
//
// The stored object keeps the layout of the unfused path ([E4M3 payload n][E8M0 scales n/32], common/mxfp8.h), and so
// does its digest: BBH64 is a sum of per-tile terms, this kernel accumulates the payload tiles (tile index 0..T-1)
// and returns the *unfinalised* sum per object; the scales region (tiles T..) is hashed as an XFER_RAW_SUM slice
// by bb_xfer and the host adds the two sums and finalises.  Objects hold any multiple of 32 elements: a tail tile is
// converted and stored like the others (its scale bytes past the last 16-byte multiple go byte-wise) but not hashed
// here -- in the packed object its hash tile also contains the first scale bytes, so the slice the host hashes simply
// starts at the last whole payload tile.
//
// Warp roles (24 warps): 0 producer, 1 MMA issuer, 2 store, 3 accumulator, 4-7 epilogue (TMEM -> row hashes),
// 8-23 convert (pack / unpack).  Two shared-memory rings: 3 x 32 KiB bf16 tiles and 6 x (16 KiB payload + 512 B scales).
#include <cuda_bf16.h>
#include <cuda_fp8.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <mutex>

#include "common/tchash_def.h"
#include "kernels/mxfp8.cuh"
#include "kernels/ptx.cuh"
#include "kernels/xfer.h"

namespace bb::gpu {
namespace {

using namespace bb::ptx;

constexpr int kWideStages = 3;              // ring of 32 KiB bf16 tiles
constexpr int kTileStages = 6;              // ring of 16 KiB payload tiles (+ 512 B scales)
constexpr int kConvertWarps = 16;           // warps 8..23 (the pack side is ALU bound: ncu issue-active 51 % with 8)
constexpr int kFpThreads = (8 + kConvertWarps) * 32;
constexpr uint32_t kWideBytes = 2 * kTileBytes;  // bf16 side of one payload tile
constexpr uint32_t kScaleBytes = kTileBytes / 32;
constexpr uint32_t kFpTmemCols = 128;       // >= kTileStages * 16 accumulator columns (power of two)
constexpr int kFpStoreLag = 1;
static_assert(kTileStages * tchash::kN <= kFpTmemCols);

__constant__ uint64_t c_fp_col_mul[tchash::kN];

struct FpMeta {            // 64 bytes
  uint64_t dst[kMaxDst];   // pack: this tile's payload address in every replica; unpack: dst[0] = bf16 destination
  int64_t scales_delta;    // pack: (tile's scales address) - (tile's payload address), the same in every replica
  uint32_t desc;
  uint32_t tile_in_obj;
  uint32_t obj_ntiles;
  uint32_t ndst;           // pack: replicas written by this pass (1..kMaxDst)
  uint32_t valid;          // payload bytes (= elements) of this tile: 16384, or the multiple-of-32 tail of the object
  uint32_t pad32;
  uint64_t pad;
};
static_assert(sizeof(FpMeta) == 64);

struct FpLookup {
  FpMeta m;
  uint64_t src;         // pack: bf16 source; unpack: payload source
  uint64_t src_scales;  // unpack: scales source
};

// Two rings: the wide (bf16) ring only spans load -> convert (pack) or convert -> store (unpack), the payload
// ring spans convert/load -> tensor-core hash -> store/accumulate.  Decoupling them lets 3 + 6 slots cover a
// pipeline that would need 6 x 48.5 KiB as one ring.
struct __align__(1024) SmemFp {
  uint8_t tile[kTileStages][kTileBytes];
  uint8_t wide[kWideStages][kWideBytes];
  uint8_t scales[kTileStages][kScaleBytes];
  uint8_t w[2048];
  uint64_t t_full[kTileStages];   // payload tile + scales ready (pack: convert warps; unpack: TMA)
  uint64_t t_empty[kTileStages];
  uint64_t w_full[kWideStages];   // wide tile ready (pack: TMA; unpack: convert warps)
  uint64_t w_empty[kWideStages];
  uint64_t acc_full[kTileStages];
  uint64_t epi_done[kTileStages];
  FpMeta t_meta[kTileStages];
  FpMeta w_meta[kWideStages];
  uint64_t part[kTileStages][4];
  FpLookup lk[32];
  uint32_t tmem_base;
};

struct FpParams {
  const XferDesc* descs;
  const uint32_t* tile_start;
  uint32_t ndesc;
  uint32_t total_tiles;
  unsigned long long* sum_ws;  // [ndesc] raw BBH64 sums of the payload tiles (zero on entry)
};

__device__ __forceinline__ uint64_t warp_sum64(uint64_t v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    uint32_t lo = __shfl_xor_sync(0xffffffffu, static_cast<uint32_t>(v), o);
    uint32_t hi = __shfl_xor_sync(0xffffffffu, static_cast<uint32_t>(v >> 32), o);
    v += (static_cast<uint64_t>(hi) << 32) | lo;
  }
  return v;
}

__device__ __forceinline__ __nv_bfloat162 as_bf162(uint32_t v) { return *reinterpret_cast<const __nv_bfloat162*>(&v); }

// One 16-byte chunk (8 bf16) per lane, 4 lanes per 32-element block.  Same arithmetic as mxfp8_pack_kernel
// (mxfp8.cu) and the CPU reference (common/mxfp8.cpp) -- the stored bytes are identical -- but on packed bf16x2
// max / paired E4M3 conversions, which halves the instruction count of the straightforward form.
__device__ __forceinline__ void pack_chunk(const uint4 v, uint2* payload_out, uint8_t* scale_out, bool write_scale) {
  // |x| on bf16x2 = clear the sign bits; max on the magnitudes as *integers* (monotonic for non-negative bf16).
  // NaN magnitudes (> 0x7F80) are skipped like the scalar code's `a > amax` does; an Inf (0x7F80) wins the max and
  // then selects the neutral scale below, again like the scalar code
  auto mag = [](uint32_t w) { return w & 0x7FFF7FFFu; };
  auto finite_max = [](uint32_t m, uint32_t cur) {
    const uint32_t lo = m & 0xFFFFu, hi = m >> 16;
    uint32_t r = cur;
    r = (lo <= 0x7F80u && lo > r) ? lo : r;
    r = (hi <= 0x7F80u && hi > r) ? hi : r;
    return r;
  };
  uint32_t am = 0;
  am = finite_max(mag(v.x), am);
  am = finite_max(mag(v.y), am);
  am = finite_max(mag(v.z), am);
  am = finite_max(mag(v.w), am);
  am = max(am, __shfl_xor_sync(0xffffffffu, am, 1));
  am = max(am, __shfl_xor_sync(0xffffffffu, am, 2));
  // am = bf16 bits of the block's largest finite magnitude; exponent field = bits 14..7
  int e = 127;
  if (am != 0 && am < 0x7F80u) {
    const int be = static_cast<int>(am >> 7);
    e = (be == 0 ? -127 : be - 127) - 8 + 127;
    e = max(0, min(254, e));
  }
  const float inv = __int_as_float((254 - e) << 23);
  auto cvt2 = [&](uint32_t w) -> uint32_t {
    const float2 f = __bfloat1622float2(as_bf162(w));
    return static_cast<uint32_t>(__nv_cvt_float2_to_fp8x2(make_float2(f.x * inv, f.y * inv), __NV_SATFINITE, __NV_E4M3));
  };
  const uint32_t lo = cvt2(v.x) | (cvt2(v.y) << 16);
  const uint32_t hi = cvt2(v.z) | (cvt2(v.w) << 16);
  *payload_out = make_uint2(lo, hi);
  if (write_scale) *scale_out = static_cast<uint8_t>(e);
}

__device__ __forceinline__ uint4 unpack_chunk(const uint2 p, uint8_t scale) {
  const float s = e8m0_scale(scale);
  auto cvt2 = [&](uint32_t two) -> uint32_t {  // two E4M3 bytes -> bf16x2
    const __half2_raw hr = __nv_cvt_fp8x2_to_halfraw2(static_cast<__nv_fp8x2_storage_t>(two & 0xFFFFu), __NV_E4M3);
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&hr));
    const __nv_bfloat162 h = __floats2bfloat162_rn(f.x * s, f.y * s);
    return *reinterpret_cast<const uint32_t*>(&h);
  };
  return make_uint4(cvt2(p.x), cvt2(p.x >> 16), cvt2(p.y), cvt2(p.y >> 16));
}

template <bool UNPACK>
__global__ void __launch_bounds__(kFpThreads, 1) bb_xfer_fp8_kernel(const __grid_constant__ FpParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  SmemFp& s = *reinterpret_cast<SmemFp*>(smem_raw);
  const uint32_t warp = threadIdx.x >> 5;
  const uint32_t lane = threadIdx.x & 31u;

  const uint32_t tpc = (p.total_tiles + gridDim.x - 1) / gridDim.x;
  const uint32_t t0 = blockIdx.x * tpc;
  const uint32_t my_tiles = t0 < p.total_tiles ? min(tpc, p.total_tiles - t0) : 0;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kTileStages; ++i) {
      mbar_init(&s.t_full[i], UNPACK ? 1 : kConvertWarps);
      mbar_init(&s.t_empty[i], UNPACK ? kConvertWarps + 1 : 2);  // unpack: convert warps + accumulator; pack: store + accumulator
      mbar_init(&s.acc_full[i], 1);
      mbar_init(&s.epi_done[i], 4);
    }
    for (int i = 0; i < kWideStages; ++i) {
      mbar_init(&s.w_full[i], UNPACK ? kConvertWarps : 1);
      mbar_init(&s.w_empty[i], UNPACK ? 1 : kConvertWarps);
    }
    fence_mbar_init();
  }
  for (uint32_t o = threadIdx.x; o < 2048; o += kFpThreads)
    s.w[o] = static_cast<uint8_t>(tchash::weight(tchash::off_to_k(o), tchash::off_to_row(o)));
  fence_proxy_async_smem();
  if (warp == 3) tmem_alloc<kFpTmemCols>(&s.tmem_base);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s.tmem_base;

  if (warp == 0) {
    // ================================================================ TMA producer
    uint32_t it = 0;
    for (uint32_t base = 0; base < my_tiles; base += 32) {
      const uint32_t idx = base + lane;
      if (idx < my_tiles) {
        const uint32_t t = t0 + idx;
        uint32_t lo = 0, hi = p.ndesc;
        while (hi - lo > 1) {
          const uint32_t mid = (lo + hi) >> 1;
          if (__ldg(&p.tile_start[mid]) <= t) lo = mid; else hi = mid;
        }
        const uint32_t first = __ldg(&p.tile_start[lo]);
        const uint32_t next = __ldg(&p.tile_start[lo + 1]);
        const uint4* q = reinterpret_cast<const uint4*>(&p.descs[lo]);
        const uint4 q0 = __ldg(q), q1 = __ldg(q + 1), q2 = __ldg(q + 2);
        const uint64_t src = (static_cast<uint64_t>(q0.y) << 32) | q0.x;
        const uint64_t d0 = (static_cast<uint64_t>(q0.w) << 32) | q0.z;
        const uint64_t d1 = (static_cast<uint64_t>(q1.y) << 32) | q1.x;
        const uint64_t d2 = (static_cast<uint64_t>(q1.w) << 32) | q1.z;
        const uint64_t nbytes = (static_cast<uint64_t>(q2.y) << 32) | q2.x;  // payload bytes == elements
        const uint32_t ti = t - first;
        FpLookup& e = s.lk[lane];
        e.m.desc = lo;
        e.m.tile_in_obj = ti;
        e.m.obj_ntiles = next - first;
        e.m.pad32 = 0;
        e.m.pad = 0;
        e.m.valid = static_cast<uint32_t>(min(static_cast<uint64_t>(kTileBytes), nbytes - static_cast<uint64_t>(ti) * kTileBytes));
        // the packed object is [payload nbytes][scales nbytes/32]: a tile's scales sit (nbytes - ti*(16384-512)) past its payload
        e.m.scales_delta = static_cast<int64_t>(nbytes) - static_cast<int64_t>(ti) * static_cast<int64_t>(kTileBytes - kScaleBytes);
        if constexpr (UNPACK) {
          e.src = src + static_cast<uint64_t>(ti) * kTileBytes;  // payload tile in the slab
          e.src_scales = e.src + e.m.scales_delta;               // its scales
          e.m.dst[0] = d0 + static_cast<uint64_t>(ti) * kWideBytes;  // bf16 destination
          e.m.dst[1] = e.m.dst[2] = 0;
          e.m.ndst = 1;
        } else {
          e.src = src + static_cast<uint64_t>(ti) * kWideBytes;  // bf16 source tile
          e.src_scales = 0;
          e.m.dst[0] = d0 + static_cast<uint64_t>(ti) * kTileBytes;
          e.m.dst[1] = d1 + static_cast<uint64_t>(ti) * kTileBytes;
          e.m.dst[2] = d2 + static_cast<uint64_t>(ti) * kTileBytes;
          e.m.ndst = min(max(q2.w, 1u), kMaxDst);
        }
      }
      __syncwarp();
      const uint32_t cnt = min(32u, my_tiles - base);
      for (uint32_t i = 0; i < cnt; ++i, ++it) {
        const FpLookup& e = s.lk[i];
        if constexpr (UNPACK) {
          const uint32_t ts = it % kTileStages, tp = (it / kTileStages) & 1u;
          mbar_wait(&s.t_empty[ts], tp ^ 1u);
          if (lane < 4) reinterpret_cast<uint4*>(&s.t_meta[ts])[lane] = reinterpret_cast<const uint4*>(&e.m)[lane];
          __syncwarp();
          // a tail tile carries valid/32 scale bytes: the 16-byte multiple by TMA, the rest byte-wise
          const uint32_t sb = e.m.valid / 32u, sb16 = sb & ~15u;
          if (lane < (sb & 15u)) s.scales[ts][sb16 + lane] = *reinterpret_cast<const uint8_t*>(e.src_scales + sb16 + lane);
          __syncwarp();
          if (lane == 0) {
            mbar_arrive_expect_tx(&s.t_full[ts], e.m.valid + sb16);
            bulk_g2s(s.tile[ts], reinterpret_cast<const void*>(e.src), e.m.valid, &s.t_full[ts]);
            if (sb16) bulk_g2s(s.scales[ts], reinterpret_cast<const void*>(e.src_scales), sb16, &s.t_full[ts]);
          }
        } else {
          const uint32_t ws = it % kWideStages, wp = (it / kWideStages) & 1u;
          mbar_wait(&s.w_empty[ws], wp ^ 1u);
          if (lane < 4) reinterpret_cast<uint4*>(&s.w_meta[ws])[lane] = reinterpret_cast<const uint4*>(&e.m)[lane];
          __syncwarp();
          if (lane == 0) {
            mbar_arrive_expect_tx(&s.w_full[ws], 2u * e.m.valid);
            bulk_g2s(s.wide[ws], reinterpret_cast<const void*>(e.src), 2u * e.m.valid, &s.w_full[ws]);
          }
        }
        __syncwarp();
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ================================================================ tensor-core hash issuer (payload tile)
    constexpr uint32_t idesc = umma_idesc_i8(tchash::kRows, tchash::kN, false, false);
    const uint32_t w_addr = smem_u32(s.w);
    for (uint32_t it = 0; it < my_tiles; ++it) {
      const uint32_t ts = it % kTileStages, tp = (it / kTileStages) & 1u;
      mbar_wait(&s.t_full[ts], tp);  // pack: written by the convert warps (generic proxy, fenced); unpack: TMA
      tc_fence_after();
      if (lane == 0) {
        const uint32_t a_addr = smem_u32(s.tile[ts]);
        const uint32_t tmem_d = tmem_base + ts * tchash::kN;
#pragma unroll
        for (uint32_t j = 0; j < tchash::kK / 32; ++j)
          mma_i8_ss(tmem_d, umma_desc_kmajor_noswizzle(a_addr + j * 256, 128, 1024), umma_desc_kmajor_noswizzle(w_addr + j * 256, 128, 1024),
                    idesc, j > 0 ? 1u : 0u);
        tc_commit(&s.acc_full[ts]);
      }
      __syncwarp();
    }
  } else if (warp == 2) {
    // ================================================================ store warp
    constexpr int kRing = UNPACK ? kWideStages : kTileStages;
    for (uint32_t it = 0; it < my_tiles; ++it) {
      const uint32_t st = it % kRing, par = (it / kRing) & 1u;
      if constexpr (UNPACK) {
        mbar_wait(&s.w_full[st], par);
        if (lane == 0) {
          bulk_s2g(reinterpret_cast<void*>(s.w_meta[st].dst[0]), s.wide[st], 2u * s.w_meta[st].valid);
          bulk_commit();
        }
      } else {
        mbar_wait(&s.t_full[st], par);
        const FpMeta& m = s.t_meta[st];
        const uint32_t sb = m.valid / 32u, sb16 = sb & ~15u;
        if (lane == 0) {
          for (uint32_t r = 0; r < m.ndst; ++r) {  // replica fan-out: converted once, stored to every copy
            bulk_s2g(reinterpret_cast<void*>(m.dst[r]), s.tile[st], m.valid);
            if (sb16) bulk_s2g(reinterpret_cast<void*>(m.dst[r] + m.scales_delta), s.scales[st], sb16);
          }
          bulk_commit();
        }
        if (lane < (sb & 15u)) {  // tail tile: the scale bytes past the last 16-byte multiple
          const uint8_t v = s.scales[st][sb16 + lane];
          for (uint32_t r = 0; r < m.ndst; ++r) *reinterpret_cast<uint8_t*>(m.dst[r] + m.scales_delta + sb16 + lane) = v;
        }
      }
      __syncwarp();
      if (it >= kFpStoreLag && lane == 0) {
        bulk_wait_read<kFpStoreLag>();
        if constexpr (UNPACK) mbar_arrive(&s.w_empty[(it - kFpStoreLag) % kRing]);
        else mbar_arrive(&s.t_empty[(it - kFpStoreLag) % kRing]);
      }
    }
    if (lane == 0) {
      bulk_wait_read<0>();
      const uint32_t first = my_tiles > kFpStoreLag ? my_tiles - kFpStoreLag : 0;
      for (uint32_t it = first; it < my_tiles; ++it) {
        if constexpr (UNPACK) mbar_arrive(&s.w_empty[it % kRing]);
        else mbar_arrive(&s.t_empty[it % kRing]);
      }
      bulk_wait<0>();
    }
  } else if (warp == 3) {
    // ================================================================ accumulator: per-object raw sums
    uint32_t cur_d = 0xFFFFFFFFu;
    uint64_t acc = 0;
    for (uint32_t it = 0; it < my_tiles; ++it) {
      const uint32_t ts = it % kTileStages, tp = (it / kTileStages) & 1u;
      mbar_wait(&s.epi_done[ts], tp);
      const uint32_t d = s.t_meta[ts].desc;
      // A tail tile holds payload AND the first scale bytes of the packed object's hash tile: it is hashed from the
      // stored bytes as part of the host's RAW_SUM slice, not here.
      const uint64_t sum = s.t_meta[ts].valid == kTileBytes ? s.part[ts][0] + s.part[ts][1] + s.part[ts][2] + s.part[ts][3] : 0;
      __syncwarp();
      if (lane == 0) mbar_arrive(&s.t_empty[ts]);
      if (d != cur_d) {
        if (cur_d != 0xFFFFFFFFu && lane == 0) atomicAdd(&p.sum_ws[cur_d], static_cast<unsigned long long>(acc));
        cur_d = d;
        acc = 0;
      }
      acc += sum;
    }
    if (cur_d != 0xFFFFFFFFu && lane == 0) atomicAdd(&p.sum_ws[cur_d], static_cast<unsigned long long>(acc));
  } else if (warp < 8) {
    // ================================================================ epilogue warps 4..7: TMEM -> row hashes
    const uint32_t q = warp & 3u;
    const uint32_t row = q * 32 + lane;
    for (uint32_t it = 0; it < my_tiles; ++it) {
      const uint32_t ts = it % kTileStages, tp = (it / kTileStages) & 1u;
      mbar_wait(&s.acc_full[ts], tp);
      mbar_wait(&s.t_full[ts], tp);  // (already complete) acquires the t_meta writes
      tc_fence_after();
      uint32_t r[16];
      tmem_ld_32x32b_x16(tmem_base + ((q * 32u) << 16) + ts * tchash::kN, r);
      tmem_ld_wait();
      tc_fence_before();
      const uint32_t ti = s.t_meta[ts].tile_in_obj;
      uint64_t rr = 0;
#pragma unroll
      for (int n = 0; n < 16; ++n) rr += static_cast<uint64_t>(r[n]) * c_fp_col_mul[n];
      const uint64_t tot = warp_sum64(tchash::row_contrib(rr, static_cast<uint64_t>(ti) * tchash::kRows + row));
      if (lane == 0) {
        s.part[ts][q] = tot;
        mbar_arrive(&s.epi_done[ts]);
      }
    }
  } else {
    // ================================================================ convert warps 8..15
    const uint32_t cw = warp - 8;  // convert warp: chunks [cw*kPer, (cw+1)*kPer) of the tile's 2048 16-byte bf16 chunks
    constexpr uint32_t kPer = 2048 / kConvertWarps;
    for (uint32_t it = 0; it < my_tiles; ++it) {
      const uint32_t ts = it % kTileStages, tp = (it / kTileStages) & 1u;
      const uint32_t ws = it % kWideStages, wp = (it / kWideStages) & 1u;
      if constexpr (UNPACK) {
        mbar_wait(&s.t_full[ts], tp);         // payload + scales landed
        mbar_wait(&s.w_empty[ws], wp ^ 1u);   // wide slot drained by the store warp
        const uint2* pay = reinterpret_cast<const uint2*>(s.tile[ts]);
        uint4* out = reinterpret_cast<uint4*>(s.wide[ws]);
#pragma unroll 4
        for (uint32_t k = 0; k < kPer / 32; ++k) {
          const uint32_t c = cw * kPer + k * 32 + lane;
          out[c] = unpack_chunk(pay[c], s.scales[ts][c >> 2]);
        }
        if (cw == 0 && lane < 4) reinterpret_cast<uint4*>(&s.w_meta[ws])[lane] = reinterpret_cast<const uint4*>(&s.t_meta[ts])[lane];
        fence_proxy_async_smem();  // generic-proxy writes -> TMA store
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(&s.w_full[ws]);
          mbar_arrive(&s.t_empty[ts]);
        }
      } else {
        mbar_wait(&s.w_full[ws], wp);         // bf16 tile landed
        mbar_wait(&s.t_empty[ts], tp ^ 1u);   // payload slot released by store + accumulator
        const uint4* in = reinterpret_cast<const uint4*>(s.wide[ws]);
        uint2* pay = reinterpret_cast<uint2*>(s.tile[ts]);
#pragma unroll 4
        for (uint32_t k = 0; k < kPer / 32; ++k) {
          const uint32_t c = cw * kPer + k * 32 + lane;
          pack_chunk(in[c], &pay[c], &s.scales[ts][c >> 2], (c & 3u) == 0);
        }
        if (cw == 0 && lane < 4) reinterpret_cast<uint4*>(&s.t_meta[ts])[lane] = reinterpret_cast<const uint4*>(&s.w_meta[ws])[lane];
        fence_proxy_async_smem();  // generic-proxy writes -> tensor core / TMA store readers
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(&s.t_full[ts]);
          mbar_arrive(&s.w_empty[ws]);
        }
      }
    }
  }

  // ------------------------------------------------------------------ teardown
  tc_fence_before();
  __syncthreads();
  if (warp == 3) {
    tc_fence_after();
    tmem_dealloc<kFpTmemCols>(tmem_base);
  }
}

struct FpDeviceState {
  bool consts = false;
  bool attr[2] = {false, false};
  int sm_count = 0;
};
FpDeviceState g_fp_dev[16];
std::mutex g_fp_mu;

}  // namespace

int xfer_fp8_smem_bytes() { return static_cast<int>(sizeof(SmemFp)); }

int launch_xfer_fp8(const XferLaunch& l, bool unpack) {
  if (l.ndesc == 0 || l.total_tiles == 0) return 0;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return static_cast<int>(e);
  if (dev < 0 || dev >= 16) return static_cast<int>(cudaErrorInvalidDevice);
  FpDeviceState& ds = g_fp_dev[dev];
  {
    std::lock_guard<std::mutex> lk(g_fp_mu);
    if (!ds.consts) {
      uint64_t h[tchash::kN];
      for (uint32_t n = 0; n < tchash::kN; ++n) h[n] = tchash::col_mul(n);
      e = cudaMemcpyToSymbol(c_fp_col_mul, h, sizeof h);
      if (e != cudaSuccess) return static_cast<int>(e);
      int n = 0;
      if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
      ds.sm_count = n;
      ds.consts = true;
    }
    if (!ds.attr[unpack ? 1 : 0]) {
      e = unpack ? cudaFuncSetAttribute(bb_xfer_fp8_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sizeof(SmemFp)))
                 : cudaFuncSetAttribute(bb_xfer_fp8_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sizeof(SmemFp)));
      if (e != cudaSuccess) return static_cast<int>(e);
      ds.attr[unpack ? 1 : 0] = true;
    }
  }
  FpParams p;
  p.descs = l.descs;
  p.tile_start = l.tile_start;
  p.ndesc = l.ndesc;
  p.total_tiles = l.total_tiles;
  p.sum_ws = reinterpret_cast<unsigned long long*>(l.sum_ws);
  int grid = l.max_ctas > 0 ? l.max_ctas : std::min(ds.sm_count, 128);
  grid = static_cast<int>(std::min<uint32_t>(static_cast<uint32_t>(grid), l.total_tiles));
  cudaStream_t st = static_cast<cudaStream_t>(l.stream);
  if (unpack) bb_xfer_fp8_kernel<true><<<grid, kFpThreads, sizeof(SmemFp), st>>>(p);
  else bb_xfer_fp8_kernel<false><<<grid, kFpThreads, sizeof(SmemFp), st>>>(p);
  return static_cast<int>(cudaGetLastError());
}

}  // namespace bb::gpu
