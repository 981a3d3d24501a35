// bb_xfer: the fused batched put/get kernel (sm_100a).
//
// Replaces the reference's per-shard UCX RMA calls (blackbird_client.cpp:231-237 put,
// :315-327 get; SURVEY K1/K4/K6/K11/K13) with ONE persistent launch per batch.  Every CTA owns
// a contiguous run of 16 KiB tiles of the batch and pipelines them through 8 smem stages:
//
//   warp 0  producer : descriptor lookup (32 tiles looked up in parallel), zero-pads short
//                      tiles, `cp.async.bulk` global -> shared (TMA, mbarrier complete_tx).
//                      The source may be local HBM (put) or a peer GPU's slab over NVLink (get).
//   warp 1  hash     : BBH64: one elected thread issues 4x `tcgen05.mma.kind::i8` (M128 N16 K32)
//                      that read the landed tile *in place* as the A operand against the BBH64
//                      weight matrix; accumulators live in TMEM (16 columns per stage).
//   warp 2  store    : `cp.async.bulk` shared -> global to 1..3 destinations (local or
//                      peer-mapped: replica fan-out with a single HBM read), or `multimem.st`
//                      to an NVLS multicast address (one store, N replicas).
//   warp 3  finalizer: folds the per-tile partials into per-object digests in registers; an
//                      object that lives entirely inside this CTA's run is finalised with no
//                      global atomics; only the <=2 objects straddling a CTA boundary use them.
//                      Compares with the expected digest on get (CHECKSUM_MISMATCH source).
//   warps 4-7 epilogue: BBH64: `tcgen05.ld` the 128x16 s32 accumulators -> position-dependent
//                      64-bit row hashes -> warp sum.  CRC32C: each warp streams its 4 KiB quarter of
//                      the tile as 8 Horner chains per lane through lane-private nibble shift tables
//                      (bank-conflict free); the chains run on across the tiles of an object and are
//                      combined (chain / lane / quarter, GF(2) shift algebra) once per object and CTA.
//
// Payload bytes never pass through registers on the BBH64 / copy-only unicast path: TMA in,
// tensor core reads shared memory, TMA out.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "common/checksum.h"
#include "common/tchash_def.h"
#include "common/xxh3.h"
#include "kernels/ptx.cuh"
#include "kernels/xfer.h"

namespace bb::gpu {
namespace {

using namespace bb::ptx;

constexpr int kStages = 8;
constexpr int kThreads = 256;
constexpr int kStoreLag = 2;         // stores may trail this many tiles before their stage is released
constexpr uint32_t kTmemCols = 128;  // kStages * 16 accumulator columns
static_assert(kStages * tchash::kN == kTmemCols);
static_assert(kTileBytes == tchash::kTileBytes);

__constant__ uint64_t c_col_mul[tchash::kN];
__constant__ uint32_t c_xpow_tiles[32];  // x^(8 * 16384 * 2^j) mod P  (CRC32C cross-CTA combine)
__constant__ uint8_t c_xxh_secret[xxh3::kSecretSize];  // XXH3 default secret

// CRC shift tables: index -> byte distance
enum CrcTab : int { T128 = 0, T4, T8, T16, T32, T64, T4096, T16384, TCHAIN, TJUMP, kNumCrcTabs };
constexpr int kCrcChains = 8;                     // independent Horner chains per lane
constexpr int kCrcChainRows = 32 / kCrcChains;   // rows (of 128 B) of a tile quarter per chain
constexpr uint64_t kCrcTabBytes[kNumCrcTabs] = {128, 4, 8, 16, 32, 64, 4096, 16384, kCrcChainRows * 128,
                                                16384 - (kCrcChainRows - 1) * 128};

struct StageMeta {  // 64 bytes
  uint64_t dst[kMaxDst];
  uint64_t nbytes;
  uint64_t expect;
  uint32_t desc;
  uint32_t tile_in_obj;
  uint32_t bytes;
  uint32_t ndst_flags;  // ndst | flags << 8
  uint32_t obj_ntiles;
  uint32_t crc_unpad;
};
static_assert(sizeof(StageMeta) == 64);

struct LookupEntry {  // producer-private staging of 32 parallel lookups
  StageMeta m;
  uint64_t src;
  uint64_t pad;
};

template <int ALGO>
struct __align__(1024) SmemT {
  uint8_t tile[kStages][kTileBytes];
  uint8_t w[2048];
  uint64_t full[kStages];
  uint64_t acc_full[kStages];
  uint64_t epi_done[kStages];
  uint64_t empty[kStages];
  StageMeta meta[kStages];
  uint64_t part[kStages][4];
  LookupEntry lk[32];
  uint32_t dirty[kStages];
  uint32_t tmem_base;
  uint32_t crc_t[ALGO == ALGO_CRC32C ? kNumCrcTabs : 1][4][256];
  // x^(8*128) shift as 8 nibble tables with one private copy per lane ([nibble][value][lane]: lane l only ever
  // touches bank l, so the 8 lookups of a step are bank-conflict free whatever the data is).
  // 2 KiB of slack: the kernel rounds the table's shared address up to 2048 so that the value index (bits 7-10)
  // can be OR-ed into the lane's base address with a single LOP3.
  uint32_t crc_nib[ALGO == ALGO_CRC32C ? 8 * 16 * 32 + 512 : 1];
  // XXH3: per-(block, lane) stripe sums of every tile in flight, written by the epilogue warps and consumed by the
  // finalizer's scramble chain; and the secret words in the order the epilogue indexes them
  // ([0..22] = accumulate keys (word s + lane), [24..31] = keys of the last stripe, [32..39] = scramble keys, [40..47] = merge keys).
  uint64_t xs[ALGO == ALGO_XXH3 ? kStages : 1][ALGO == ALGO_XXH3 ? 16 : 1][8];
  uint64_t xkey[ALGO == ALGO_XXH3 ? 48 : 1];
};

struct Params {
  const XferDesc* descs;
  const uint32_t* tile_start;
  uint32_t ndesc;
  uint32_t total_tiles;
  unsigned long long* sum_ws;
  uint32_t* done_ws;
  uint64_t* digest_out;
  uint32_t* status_out;
  const uint32_t* crc_tables;  // [kNumCrcTabs][4][256]
  uint32_t* debug_d;
  // Optional per-tile pipeline trace (diagnostics): [tile][4] globaltimer ns = load issued, tile landed in smem,
  // store issued, smem slot released.
  unsigned long long* trace_d;
  // Small batches carry their descriptor table in the kernel parameters (constant bank): no H2D
  // copy ahead of the launch, which is most of a single-object put/get's latency.
  uint32_t use_inline;
  uint32_t inl_tile_start[kInlineDescs + 1];
  XferDesc inl_descs[kInlineDescs];
};

__device__ __forceinline__ uint64_t shfl_xor_u64(uint64_t v, int m) {
  const uint32_t lo = __shfl_xor_sync(0xffffffffu, static_cast<uint32_t>(v), m);
  const uint32_t hi = __shfl_xor_sync(0xffffffffu, static_cast<uint32_t>(v >> 32), m);
  return (static_cast<uint64_t>(hi) << 32) | lo;
}
__device__ __forceinline__ uint64_t shfl_u64(uint64_t v, int src) {
  const uint32_t lo = __shfl_sync(0xffffffffu, static_cast<uint32_t>(v), src);
  const uint32_t hi = __shfl_sync(0xffffffffu, static_cast<uint32_t>(v >> 32), src);
  return (static_cast<uint64_t>(hi) << 32) | lo;
}

__device__ __forceinline__ uint64_t warp_sum64(uint64_t v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    uint32_t lo = __shfl_xor_sync(0xffffffffu, static_cast<uint32_t>(v), o);
    uint32_t hi = __shfl_xor_sync(0xffffffffu, static_cast<uint32_t>(v >> 32), o);
    v += (static_cast<uint64_t>(hi) << 32) | lo;
  }
  return v;
}

// s * x^(8k) mod P through the 4x256 table of distance k.
__device__ __forceinline__ uint32_t crc_shift(const uint32_t (*t)[256], uint32_t s) {
  return t[0][s & 0xFFu] ^ t[1][(s >> 8) & 0xFFu] ^ t[2][(s >> 16) & 0xFFu] ^ t[3][s >> 24];
}

// One nibble of the lane-private x^(8*128) shift: table [nibble J][value][lane], 2 KiB per nibble, base 2 KiB aligned
// so the value index (bits 7-10) is OR-ed into the lane's base address by one LOP3.  The table is read-only after setup.
template <int J>
__device__ __forceinline__ uint32_t crc_nib_lookup(uint32_t v, uint32_t nib_lane) {
  const uint32_t x = (4 * J >= 7) ? (v >> (4 * J >= 7 ? 4 * J - 7 : 0)) : (v << (4 * J >= 7 ? 0 : 7 - 4 * J));
  uint32_t addr, t;
  asm("lop3.b32 %0, %1, 0x780, %2, 0xEA;" : "=r"(addr) : "r"(x), "r"(nib_lane));  // (x & 0x780) | base
  asm("ld.shared.u32 %0, [%1+%2];" : "=r"(t) : "r"(addr), "n"(J * 2048));
  return t;
}
__device__ __forceinline__ uint32_t crc_nib_shift(uint32_t v, uint32_t nib_lane) {
  return crc_nib_lookup<0>(v, nib_lane) ^ crc_nib_lookup<1>(v, nib_lane) ^ crc_nib_lookup<2>(v, nib_lane) ^
         crc_nib_lookup<3>(v, nib_lane) ^ crc_nib_lookup<4>(v, nib_lane) ^ crc_nib_lookup<5>(v, nib_lane) ^
         crc_nib_lookup<6>(v, nib_lane) ^ crc_nib_lookup<7>(v, nib_lane);
}

__device__ __forceinline__ uint32_t gf2_mulmod_dev(uint32_t a, uint32_t b) {
  uint32_t p = 0;
#pragma unroll 4
  for (int i = 31; i >= 0; --i) {
    p ^= ((a >> i) & 1u) ? b : 0u;
    b = (b >> 1) ^ ((b & 1u) ? 0x82F63B78u : 0u);
  }
  return p;
}

// x^(8*16384*k) mod P, computed cooperatively by a full warp (lane j owns bit j of k).
__device__ __forceinline__ uint32_t warp_xpow_tiles(uint32_t k, uint32_t lane) {
  uint32_t v = ((k >> lane) & 1u) ? c_xpow_tiles[lane] : 0x80000000u;  // 0x80000000 == 1
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const uint32_t other = __shfl_xor_sync(0xffffffffu, v, o);
    v = gf2_mulmod_dev(v, other);
  }
  return v;
}

// Segment tables (XferSeg, kernels/xfer.h).  Index j >= 1 of the first segment whose end lies past `off`.
__device__ __forceinline__ uint32_t seg_find(const XferSeg* t, uint64_t off) {
  uint32_t lo = 1, hi = static_cast<uint32_t>(__ldg(&t[0].addr));
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (__ldg(&t[mid].end) > off) hi = mid; else lo = mid + 1;
  }
  return lo;
}
// Address of object byte `off`, which lies in the table's last segment (the byte tail of an object).
__device__ __forceinline__ uint64_t seg_last_addr(const XferSeg* t, uint64_t off) {
  const uint32_t n = static_cast<uint32_t>(__ldg(&t[0].addr));
  return __ldg(&t[n].addr) + (off - __ldg(&t[n - 1].end));
}
// Calls f(global address, tile offset, bytes) once per piece of the 16-byte part [off, off + b16) of a tile, starting at
// segment `first` (seg_find).  The pieces are spread over the lanes of the warp: lane l takes segments first + l,
// first + l + 32, ...  Every piece is 16-byte aligned and a multiple of 16 bytes long (the segment rules).
template <typename F>
__device__ __forceinline__ void seg_pieces(const XferSeg* t, uint32_t first, uint64_t off, uint32_t b16, uint32_t lane, F&& f) {
  if (b16 == 0) return;
  const uint32_t n = static_cast<uint32_t>(__ldg(&t[0].addr));
  const uint64_t lim = off + b16;
  for (uint32_t j0 = first;; j0 += 32) {
    const uint32_t j = j0 + lane;
    bool more = false;
    if (j <= n) {
      const uint64_t sb = __ldg(&t[j - 1].end);
      if (sb < lim) {
        const uint64_t se = __ldg(&t[j].end);
        const uint64_t lo = sb > off ? sb : off, hi = se < lim ? se : lim;
        f(__ldg(&t[j].addr) + (lo - sb), static_cast<uint32_t>(lo - off), static_cast<uint32_t>(hi - lo));
        more = true;
      }
    }
    if (!__shfl_sync(0xffffffffu, more ? 1u : 0u, 31)) break;
  }
}

template <int ALGO, bool SEG>
__global__ void __launch_bounds__(kThreads, 1) bb_xfer_kernel(const __grid_constant__ Params p) {
  using Smem = SmemT<ALGO>;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  Smem& s = *reinterpret_cast<Smem*>(smem_raw);
  const uint32_t warp = threadIdx.x >> 5;
  const uint32_t lane = threadIdx.x & 31u;
  constexpr bool kBbh = (ALGO == ALGO_BBH64);
  constexpr bool kCrc = (ALGO == ALGO_CRC32C);
  constexpr bool kXxh = (ALGO == ALGO_XXH3);
  constexpr bool kSum = kBbh || kXxh;  // digest = finalize(commutative sum of per-tile terms)
  constexpr bool kHash = kBbh || kCrc || kXxh;

  // contiguous run of tiles for this CTA
  const uint32_t tpc = (p.total_tiles + gridDim.x - 1) / gridDim.x;
  const uint32_t t0 = blockIdx.x * tpc;
  const uint32_t my_tiles = t0 < p.total_tiles ? min(tpc, p.total_tiles - t0) : 0;

  // ------------------------------------------------------------------ setup
  if (threadIdx.x == 0) {
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&s.full[i], 1);
      mbar_init(&s.acc_full[i], 1);
      mbar_init(&s.epi_done[i], 4);
      mbar_init(&s.empty[i], kHash ? 2 : 1);  // store warp (+ finalizer)
      s.dirty[i] = kTileBytes;
    }
    fence_mbar_init();
  }
  if constexpr (kBbh) {
    // BBH64 weight matrix W[k][n] as the UMMA B operand (N=16 rows, K-major, no swizzle).
    for (uint32_t o = threadIdx.x; o < 2048; o += kThreads)
      s.w[o] = static_cast<uint8_t>(tchash::weight(tchash::off_to_k(o), tchash::off_to_row(o)));
    fence_proxy_async_smem();
    if (warp == 3) tmem_alloc<kTmemCols>(&s.tmem_base);
    tc_fence_before();
  }
  if constexpr (kCrc) {
    uint32_t* dstt = &s.crc_t[0][0][0];
    for (uint32_t i = threadIdx.x; i < kNumCrcTabs * 1024; i += kThreads) dstt[i] = __ldg(&p.crc_tables[i]);
    __syncthreads();
    uint32_t* nibt = s.crc_nib + ((2048u - (smem_u32(s.crc_nib) & 2047u)) & 2047u) / 4u;
    for (uint32_t i = threadIdx.x; i < 8 * 16 * 32; i += kThreads) {  // [nibble j][value v][lane]
      const uint32_t j = i >> 9, v = (i >> 5) & 15u;
      nibt[i] = crc_shift(s.crc_t[T128], v << (4 * j));
    }
  }
  if constexpr (kXxh) {
    if (threadIdx.x < 48) {
      const uint32_t i = threadIdx.x;
      uint64_t v = 0;
      const uint32_t off = i < 24 ? 8u * min(i, 22u) : i < 32 ? xxh3::kSecretSize - xxh3::kStripe - xxh3::kLastAccStart + 8u * (i - 24)
                           : i < 40 ? xxh3::kSecretSize - xxh3::kStripe + 8u * (i - 32) : xxh3::kMergeStart + 8u * (i - 40);
      for (int b = 7; b >= 0; --b) v = (v << 8) | c_xxh_secret[off + b];
      s.xkey[i] = v;
    }
  }
  __syncthreads();
  if constexpr (kBbh) tc_fence_after();
  const uint32_t tmem_base = kBbh ? s.tmem_base : 0;

  if (warp == 0) {
    // ================================================================ TMA producer
    uint32_t it = 0;
    for (uint32_t base = 0; base < my_tiles; base += 32) {
      const uint32_t idx = base + lane;
      if (idx < my_tiles) {
        const uint32_t t = t0 + idx;
        uint32_t lo = 0, hi = p.ndesc;  // tile_start[lo] <= t < tile_start[hi]
        uint32_t first, next;
        uint4 q0, q1, q2, q3;
        if (!SEG && p.use_inline) {  // table in the parameter space (plain loads: ld.global.nc is illegal there)
          while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (p.inl_tile_start[mid] <= t) lo = mid; else hi = mid;
          }
          first = p.inl_tile_start[lo];
          next = p.inl_tile_start[lo + 1];
          const uint4* q = reinterpret_cast<const uint4*>(&p.inl_descs[lo]);
          q0 = q[0], q1 = q[1], q2 = q[2], q3 = q[3];
        } else {
          while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (__ldg(&p.tile_start[mid]) <= t) lo = mid; else hi = mid;
          }
          first = __ldg(&p.tile_start[lo]);
          next = __ldg(&p.tile_start[lo + 1]);
          const uint4* q = reinterpret_cast<const uint4*>(&p.descs[lo]);
          q0 = __ldg(q), q1 = __ldg(q + 1), q2 = __ldg(q + 2), q3 = __ldg(q + 3);
        }
        LookupEntry& e = s.lk[lane];
        e.src = (static_cast<uint64_t>(q0.y) << 32) | q0.x;
        e.m.dst[0] = (static_cast<uint64_t>(q0.w) << 32) | q0.z;
        e.m.dst[1] = (static_cast<uint64_t>(q1.y) << 32) | q1.x;
        e.m.dst[2] = (static_cast<uint64_t>(q1.w) << 32) | q1.z;
        e.m.nbytes = (static_cast<uint64_t>(q2.y) << 32) | q2.x;
        e.m.expect = (static_cast<uint64_t>(q3.y) << 32) | q3.x;
        e.m.desc = lo;
        e.m.tile_in_obj = t - first;
        e.m.ndst_flags = (q2.w & 0xFFu) | (q3.z << 8);
        e.m.obj_ntiles = next - first;
        e.m.crc_unpad = q3.w;
        if constexpr (SEG) {
          // first segment of this tile, looked up for 32 tiles at once: the gather index rides in the entry's spare word,
          // the scatter index in dst[1] (a scatter descriptor has one destination)
          const uint64_t toff = static_cast<uint64_t>(t - first) * kTileBytes;
          if (q3.z & XFER_GATHER) e.pad = seg_find(reinterpret_cast<const XferSeg*>(e.src), toff);
          if (q3.z & XFER_SCATTER) e.m.dst[1] = seg_find(reinterpret_cast<const XferSeg*>(e.m.dst[0]), toff);
        }
      }
      __syncwarp();
      const uint32_t cnt = min(32u, my_tiles - base);
      for (uint32_t i = 0; i < cnt; ++i, ++it) {
        const uint32_t stage = it % kStages;
        const uint32_t par = (it / kStages) & 1u;
        const LookupEntry& e = s.lk[i];
        const uint64_t src_i = e.src;
        const uint64_t off = static_cast<uint64_t>(e.m.tile_in_obj) * kTileBytes;
        const uint32_t bytes = static_cast<uint32_t>(min(static_cast<uint64_t>(kTileBytes), e.m.nbytes - off));
        const uint32_t b16 = bytes & ~15u;
        const uint32_t tail = bytes & 15u;
        const bool gather = SEG && ((e.m.ndst_flags >> 8) & XFER_GATHER);
        mbar_wait(&s.empty[stage], par ^ 1u);
        bool wrote = false;
        if constexpr (kHash) {
          const uint32_t dirty = s.dirty[stage];
          for (uint32_t o = b16 + lane * 16; o < dirty; o += 512) {
            *reinterpret_cast<uint4*>(&s.tile[stage][o]) = make_uint4(0, 0, 0, 0);
            wrote = true;
          }
        }
        if (lane < tail) {
          if constexpr (SEG) {
            const uint64_t a = gather ? seg_last_addr(reinterpret_cast<const XferSeg*>(src_i), off + b16) : src_i + off + b16;
            s.tile[stage][b16 + lane] = *reinterpret_cast<const uint8_t*>(a + lane);
          } else {
            s.tile[stage][b16 + lane] = *reinterpret_cast<const uint8_t*>(src_i + off + b16 + lane);
          }
          wrote = true;
        }
        if (wrote) fence_proxy_async_smem();
        if (lane < 4) {
          uint4 v = reinterpret_cast<const uint4*>(&e.m)[lane];
          if (lane == 3) v.x = bytes;  // StageMeta::bytes is the first word of uint4 #3
          reinterpret_cast<uint4*>(&s.meta[stage])[lane] = v;
        }
        __syncwarp();
        if (lane == 0) {
          s.dirty[stage] = (bytes + 15u) & ~15u;
          mbar_arrive_expect_tx(&s.full[stage], b16);
          if (b16 && !gather) bulk_g2s(s.tile[stage], reinterpret_cast<const void*>(src_i + off), b16, &s.full[stage]);
          if (p.trace_d) p.trace_d[static_cast<uint64_t>(t0 + base + i) * 4 + 0] = globaltimer_ns();
        }
        if constexpr (SEG) {
          if (gather) {  // one bulk copy per piece, all completing on the stage's barrier (armed above with the b16 total)
            __syncwarp();
            const uint32_t first = static_cast<uint32_t>(e.pad);
            seg_pieces(reinterpret_cast<const XferSeg*>(src_i), first, off, b16, lane, [&](uint64_t g, uint32_t to, uint32_t nb) {
              bulk_g2s(&s.tile[stage][to], reinterpret_cast<const void*>(g), nb, &s.full[stage]);
            });
          }
        }
        __syncwarp();
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ================================================================ tensor-core hash issuer
    if constexpr (kBbh) {
      constexpr uint32_t idesc = umma_idesc_i8(tchash::kRows, tchash::kN, false, false);
      const uint32_t w_addr = smem_u32(s.w);
      for (uint32_t it = 0; it < my_tiles; ++it) {
        const uint32_t stage = it % kStages;
        const uint32_t par = (it / kStages) & 1u;
        mbar_wait(&s.full[stage], par);
        tc_fence_after();
        if (lane == 0) {
          const uint32_t a_addr = smem_u32(s.tile[stage]);
          const uint32_t tmem_d = tmem_base + stage * tchash::kN;
#pragma unroll
          for (uint32_t j = 0; j < tchash::kK / 32; ++j) {
            // each MMA consumes K=32 bytes = two 16-byte K chunks (LBO 128 B apart)
            mma_i8_ss(tmem_d, umma_desc_kmajor_noswizzle(a_addr + j * 256, 128, 1024),
                      umma_desc_kmajor_noswizzle(w_addr + j * 256, 128, 1024), idesc, j > 0 ? 1u : 0u);
          }
          tc_commit(&s.acc_full[stage]);
        }
        __syncwarp();
      }
    }
  } else if (warp == 2) {
    // ================================================================ store warp
    for (uint32_t it = 0; it < my_tiles; ++it) {
      const uint32_t stage = it % kStages;
      const uint32_t par = (it / kStages) & 1u;
      mbar_wait(&s.full[stage], par);
      if (p.trace_d && lane == 0) p.trace_d[static_cast<uint64_t>(t0 + it) * 4 + 1] = globaltimer_ns();
      const StageMeta& m = s.meta[stage];
      const uint64_t off = static_cast<uint64_t>(m.tile_in_obj) * kTileBytes;
      const uint32_t b16 = m.bytes & ~15u;
      const uint32_t tail = m.bytes & 15u;
      const uint32_t ndst = m.ndst_flags & 0xFFu;
      const uint32_t flags = m.ndst_flags >> 8;
      // scatter: dst[0] is the segment table, dst[1] the first segment of this tile; any lane may issue a piece, so in
      // the segmented kernel every lane keeps its own bulk groups (commit / wait below)
      const bool scatter = SEG && (flags & XFER_SCATTER);
      if (flags & XFER_MULTIMEM) {
        uint8_t* mc = reinterpret_cast<uint8_t*>(m.dst[0] + off);
        for (uint32_t o = lane * 16; o < b16; o += 512)
          multimem_st_v4(mc + o, *reinterpret_cast<const uint4*>(&s.tile[stage][o]));
      } else if (scatter) {
        seg_pieces(reinterpret_cast<const XferSeg*>(m.dst[0]), static_cast<uint32_t>(m.dst[1]), off, b16, lane,
                   [&](uint64_t g, uint32_t to, uint32_t nb) { bulk_s2g(reinterpret_cast<void*>(g), &s.tile[stage][to], nb); });
      } else if (lane == 0) {
        for (uint32_t r = 0; r < ndst; ++r)
          if (b16) bulk_s2g(reinterpret_cast<void*>(m.dst[r] + off), s.tile[stage], b16);
      }
      if (SEG || lane == 0) bulk_commit();
      if (p.trace_d && lane == 0) p.trace_d[static_cast<uint64_t>(t0 + it) * 4 + 2] = globaltimer_ns();
      if (lane < tail) {
        const uint8_t b = s.tile[stage][b16 + lane];
        if (scatter) {
          *reinterpret_cast<uint8_t*>(seg_last_addr(reinterpret_cast<const XferSeg*>(m.dst[0]), off + b16) + lane) = b;
        } else {
          for (uint32_t r = 0; r < ndst; ++r) *reinterpret_cast<uint8_t*>(m.dst[r] + off + b16 + lane) = b;
        }
      }
      __syncwarp();
      if constexpr (SEG) {
        if (it >= kStoreLag) {
          bulk_wait_read<kStoreLag>();
          __syncwarp();
          if (lane == 0) {
            mbar_arrive(&s.empty[(it - kStoreLag) % kStages]);
            if (p.trace_d) p.trace_d[static_cast<uint64_t>(t0 + it - kStoreLag) * 4 + 3] = globaltimer_ns();
          }
        }
      } else {
        if (it >= kStoreLag && lane == 0) {
          bulk_wait_read<kStoreLag>();
          mbar_arrive(&s.empty[(it - kStoreLag) % kStages]);
          if (p.trace_d) p.trace_d[static_cast<uint64_t>(t0 + it - kStoreLag) * 4 + 3] = globaltimer_ns();
        }
      }
    }
    if constexpr (SEG) {
      bulk_wait_read<0>();
      __syncwarp();
    }
    if (lane == 0) {
      bulk_wait_read<0>();
      const uint32_t first = my_tiles > kStoreLag ? my_tiles - kStoreLag : 0;
      for (uint32_t it = first; it < my_tiles; ++it) {
        mbar_arrive(&s.empty[it % kStages]);
        if (p.trace_d) p.trace_d[static_cast<uint64_t>(t0 + it) * 4 + 3] = globaltimer_ns();
      }
      bulk_wait<0>();  // writes performed before the kernel retires
    }
    if constexpr (SEG) bulk_wait<0>();
  } else if (warp == 3) {
    // ================================================================ finalizer
    if constexpr (kHash) {
      uint32_t cur_d = 0xFFFFFFFFu, cnt = 0;
      uint64_t acc = 0;
      // Folds one finished tile (its StageMeta `m` and the epilogue's partials) into the running per-object state and,
      // when this CTA's share of the object is complete, publishes / combines it.
      auto account = [&](uint32_t it, const StageMeta& m, uint64_t p0, uint64_t p1, uint64_t p2, uint64_t p3) {
        if (m.desc != cur_d) {
          cur_d = m.desc;
          acc = 0;
          cnt = 0;
        }
        if constexpr (kSum) acc += p0 + p1 + p2 + p3;
        ++cnt;
        const bool obj_end = (m.tile_in_obj + 1 == m.obj_ntiles);
        if (obj_end || it + 1 == my_tiles) {
          if constexpr (kCrc) {
            // The epilogue warps carry their per-lane accumulators across the tiles of an object and publish the
            // four quarter values only here: together they are the CRC polynomial of this CTA's whole run of it.
            const auto* t4k = s.crc_t[T4096];
            uint32_t t = crc_shift(t4k, static_cast<uint32_t>(p0)) ^ static_cast<uint32_t>(p1);
            t = crc_shift(t4k, t) ^ static_cast<uint32_t>(p2);
            t = crc_shift(t4k, t) ^ static_cast<uint32_t>(p3);
            acc = t;
          }
          // ---- this CTA's contribution to object cur_d is complete
          uint64_t digest = 0;
          bool have = false;
          const bool raw = kSum && ((m.ndst_flags >> 8) & XFER_RAW_SUM);
          if (cnt == m.obj_ntiles) {  // object lives entirely in this CTA: no atomics
            if constexpr (kSum) digest = raw ? acc : tchash::finalize(acc, m.nbytes);
            else digest = gf2_mulmod_dev(static_cast<uint32_t>(acc), m.crc_unpad) ^ static_cast<uint32_t>(m.expect >> 32) ^ 0xFFFFFFFFu;
            have = true;
          } else {
            uint64_t contrib = acc;
            if constexpr (kCrc) {
              const uint32_t after = m.obj_ntiles - 1u - m.tile_in_obj;  // tiles of this object after my run
              contrib = gf2_mulmod_dev(static_cast<uint32_t>(acc), warp_xpow_tiles(after, lane));
            }
            uint32_t prev = 0;
            if (lane == 0) {
              if constexpr (kSum) atomicAdd(&p.sum_ws[cur_d], static_cast<unsigned long long>(contrib));
              else atomicXor(&p.sum_ws[cur_d], static_cast<unsigned long long>(contrib));
              __threadfence();
              prev = atomicAdd(&p.done_ws[cur_d], cnt);
            }
            prev = __shfl_sync(0xffffffffu, prev, 0);
            if (prev + cnt == m.obj_ntiles) {  // last contributor finalises and re-zeroes
              if (lane == 0) {
                __threadfence();
                const uint64_t sum = atomicExch(&p.sum_ws[cur_d], 0ull);
                p.done_ws[cur_d] = 0;
                if constexpr (kSum) digest = raw ? sum : tchash::finalize(sum, m.nbytes);
                else digest = gf2_mulmod_dev(static_cast<uint32_t>(sum), m.crc_unpad) ^ static_cast<uint32_t>(m.expect >> 32) ^ 0xFFFFFFFFu;
              }
              have = true;
            }
          }
          if (have && lane == 0) {
            const uint64_t want = kSum ? m.expect : (m.expect & 0xFFFFFFFFull);
            p.digest_out[cur_d] = digest;
            p.status_out[cur_d] = (((m.ndst_flags >> 8) & XFER_VERIFY) && digest != want) ? 1u : 0u;
          }
          cur_d = 0xFFFFFFFFu;
        }
      };
      if constexpr (kXxh) {
        // XXH3: the epilogue warps left the 16 x 8 (block, lane) stripe sums of each tile in s.xs; what remains is the
        // serial part of the algorithm -- 15 scrambles per accumulator lane, then the merge.  The chain is latency bound
        // (~40 dependent cycles per step), so four tiles are chained at once, one per group of 8 lanes.
        const uint32_t g = lane >> 3, l8 = lane & 7u;
        const uint64_t skey = s.xkey[32 + l8], mkey = s.xkey[40 + l8];
        for (uint32_t it0 = 0; it0 < my_tiles; it0 += 4) {
          const uint32_t n = min(4u, my_tiles - it0);
          for (uint32_t j = 0; j < n; ++j) mbar_wait(&s.epi_done[(it0 + j) % kStages], ((it0 + j) / kStages) & 1u);
          const uint32_t st = (it0 + min(g, n - 1u)) % kStages;  // idle groups redo the last tile (their result is ignored)
          uint64_t a = xxh3::init_acc(l8);
#pragma unroll
          for (int b = 0; b < 15; ++b) a = xxh3::scramble(a + s.xs[st][b][l8], skey);
          a += s.xs[st][15][l8];
          const uint64_t nb = shfl_u64(a, static_cast<int>((lane + 1u) & 31u));  // the odd lane's accumulator and key
          const uint64_t nk = shfl_u64(mkey, static_cast<int>((lane + 1u) & 31u));
          uint64_t mg = (l8 & 1u) ? 0ull : xxh3::mul128_fold64(a ^ mkey, nb ^ nk);
          mg += shfl_xor_u64(mg, 2);
          mg += shfl_xor_u64(mg, 4);
          const uint64_t h = xxh3::avalanche(mg + static_cast<uint64_t>(kTileBytes) * xxh3::P64_1);  // XXH3_64bits(tile), in lanes l8 == 0
          __syncwarp();
          for (uint32_t j = 0; j < n; ++j) {
            const uint32_t stage = (it0 + j) % kStages;
            const StageMeta m = s.meta[stage];
            const uint64_t hj = shfl_u64(h, static_cast<int>(j * 8u));
            __syncwarp();
            if (lane == 0) mbar_arrive(&s.empty[stage]);
            const uint32_t ti = m.tile_in_obj + (((m.ndst_flags >> 8) & XFER_RAW_SUM) ? m.crc_unpad : 0u);
            account(it0 + j, m, tchash::mix64(hj + (static_cast<uint64_t>(ti) + 1ull) * tchash::kGold), 0, 0, 0);
          }
        }
      } else {
        for (uint32_t it = 0; it < my_tiles; ++it) {
          const uint32_t stage = it % kStages;
          const uint32_t par = (it / kStages) & 1u;
          mbar_wait(&s.epi_done[stage], par);
          const StageMeta m = s.meta[stage];
          const uint64_t p0 = s.part[stage][0], p1 = s.part[stage][1], p2 = s.part[stage][2], p3 = s.part[stage][3];
          __syncwarp();
          if (lane == 0) mbar_arrive(&s.empty[stage]);
          account(it, m, p0, p1, p2, p3);
        }
      }
    }
  } else {
    // ================================================================ epilogue warps 4..7
    if constexpr (kBbh) {
      const uint32_t q = warp & 3u;
      const uint32_t row = q * 32 + lane;
      for (uint32_t it = 0; it < my_tiles; ++it) {
        const uint32_t stage = it % kStages;
        const uint32_t par = (it / kStages) & 1u;
        mbar_wait(&s.acc_full[stage], par);
        mbar_wait(&s.full[stage], par);  // already complete; acquires the producer's StageMeta writes
        tc_fence_after();
        uint32_t r[16];
        tmem_ld_32x32b_x16(tmem_base + ((q * 32u) << 16) + stage * tchash::kN, r);
        tmem_ld_wait();
        tc_fence_before();
        // position of this tile in the hashed object (a RAW_SUM slice starts at a non-zero tile index)
        const uint32_t ti = s.meta[stage].tile_in_obj + (((s.meta[stage].ndst_flags >> 8) & XFER_RAW_SUM) ? s.meta[stage].crc_unpad : 0u);
        uint64_t rr = 0;
#pragma unroll
        for (int n = 0; n < 16; ++n) rr += static_cast<uint64_t>(r[n]) * c_col_mul[n];
        const uint64_t tot = warp_sum64(tchash::row_contrib(rr, static_cast<uint64_t>(ti) * tchash::kRows + row));
        if (lane == 0) {
          s.part[stage][q] = tot;
          mbar_arrive(&s.epi_done[stage]);
        }
        if (p.debug_d) {
          uint32_t* o = p.debug_d + (static_cast<uint64_t>(t0 + it) * tchash::kRows + row) * tchash::kN;
#pragma unroll
          for (int n = 0; n < 16; ++n) o[n] = r[n];
        }
      }
    } else if constexpr (kXxh) {
      // XXH3 stripe sums.  A block's 16 stripe contributions do not depend on the accumulator, so all 16 x 8 (block,
      // lane) sums of the tile are computed at once: quarter-warp = one 1 KiB block, thread = (lane pair, half of the
      // stripes), one LDS.128 per stripe = the two 8-byte lanes of the pair (so the "swap" addend stays in the thread).
      // The odd half visits its stripes shifted by one: the 8 threads of a quarter then cover all 32 banks every time.
      const uint32_t e = threadIdx.x - 128u;
      const uint32_t blk = (e >> 5) * 4u + ((e & 31u) >> 3);
      const uint32_t pair = (e >> 1) & 3u, half = e & 1u;
      for (uint32_t it = 0; it < my_tiles; ++it) {
        const uint32_t stage = it % kStages;
        const uint32_t par = (it / kStages) & 1u;
        mbar_wait(&s.full[stage], par);
        const uint8_t* base = &s.tile[stage][blk * 1024u + pair * 16u];
        uint64_t s0 = 0, s1 = 0;
#pragma unroll
        for (uint32_t k = 0; k < 8; ++k) {
          const uint32_t stp = half * 8u + ((k + half) & 7u);
          const uint4 d = *reinterpret_cast<const uint4*>(base + stp * 64u);
          const uint64_t dv0 = (static_cast<uint64_t>(d.y) << 32) | d.x, dv1 = (static_cast<uint64_t>(d.w) << 32) | d.z;
          const uint32_t ki = (blk == 15u && stp == 15u) ? 24u + 2u * pair : stp + 2u * pair;  // the tile's very last stripe has its own key
          const uint64_t q0 = dv0 ^ s.xkey[ki], q1 = dv1 ^ s.xkey[ki + 1u];
          s0 += static_cast<uint64_t>(static_cast<uint32_t>(q0)) * (q0 >> 32) + dv1;
          s1 += static_cast<uint64_t>(static_cast<uint32_t>(q1)) * (q1 >> 32) + dv0;
        }
        s0 += shfl_xor_u64(s0, 1);
        s1 += shfl_xor_u64(s1, 1);
        if (half == 0u) {
          s.xs[stage][blk][2u * pair] = s0;
          s.xs[stage][blk][2u * pair + 1u] = s1;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&s.epi_done[stage]);
      }
    } else if constexpr (kCrc) {
      // Quarter q of every tile, lane l: words l, l+32, ... (bank-conflict free); consecutive words of a lane are
      // 128 B apart -> one x^(8*128) shift per step through the lane-private nibble tables.  Four independent Horner
      // chains per lane (kCrcChains x kCrcChainRows rows) hide the latency of the dependent lookups, and the chains
      // run on ACROSS the tiles of an object (a chain's next row in the following tile is 16384 - (kCrcChainRows-1)*128 bytes
      // further), so the lane / chain / quarter combine is paid once per object and CTA, not once per tile.
      const uint32_t q = warp & 3u;
      const uint32_t nib_lane = ((smem_u32(s.crc_nib) + 2047u) & ~2047u) + lane * 4u;  // bits 7-10 clear
      const auto* tj = s.crc_t[TJUMP];
      uint32_t a[kCrcChains];
#pragma unroll
      for (int c = 0; c < kCrcChains; ++c) a[c] = 0;
      for (uint32_t it = 0; it < my_tiles; ++it) {
        const uint32_t stage = it % kStages;
        const uint32_t par = (it / kStages) & 1u;
        mbar_wait(&s.full[stage], par);  // also acquires the producer's StageMeta writes
        const uint32_t tio = s.meta[stage].tile_in_obj;
        const bool fresh = (it == 0) || (tio == 0);
        const bool flush = (tio + 1 == s.meta[stage].obj_ntiles) || (it + 1 == my_tiles);
        const uint32_t* wp = reinterpret_cast<const uint32_t*>(&s.tile[stage][q * 4096]) + lane;
        if (fresh) {
#pragma unroll
          for (int c = 0; c < kCrcChains; ++c) a[c] = wp[c * kCrcChainRows * 32];
        } else {
#pragma unroll
          for (int c = 0; c < kCrcChains; ++c) a[c] = crc_shift(tj, a[c]) ^ wp[c * kCrcChainRows * 32];
        }
#pragma unroll
        for (int i = 1; i < kCrcChainRows; ++i) {
#pragma unroll
          for (int c = 0; c < kCrcChains; ++c) a[c] = crc_nib_shift(a[c], nib_lane) ^ wp[(c * kCrcChainRows + i) * 32];
        }
        if (flush) {
          const auto* tc = s.crc_t[TCHAIN];  // chains are kCrcChainRows rows of 128 B apart
          uint32_t v = a[0];
#pragma unroll
          for (int c = 1; c < kCrcChains; ++c) v = crc_shift(tc, v) ^ a[c];
          // combine lanes: value(l) covers bytes [4l, 4l+4) of each 128-byte row group
          uint32_t o;
          o = __shfl_down_sync(0xffffffffu, v, 1);  v = crc_shift(s.crc_t[T4], v) ^ o;
          o = __shfl_down_sync(0xffffffffu, v, 2);  v = crc_shift(s.crc_t[T8], v) ^ o;
          o = __shfl_down_sync(0xffffffffu, v, 4);  v = crc_shift(s.crc_t[T16], v) ^ o;
          o = __shfl_down_sync(0xffffffffu, v, 8);  v = crc_shift(s.crc_t[T32], v) ^ o;
          o = __shfl_down_sync(0xffffffffu, v, 16); v = crc_shift(s.crc_t[T64], v) ^ o;
          if (lane == 0) s.part[stage][q] = crc_shift(s.crc_t[T4], v);  // the CRC's final x^32 factor
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&s.epi_done[stage]);
      }
    }
  }

  // ------------------------------------------------------------------ teardown
  if constexpr (kBbh) tc_fence_before();
  __syncthreads();
  if constexpr (kBbh) {
    if (warp == 3) {
      tc_fence_after();
      tmem_dealloc<kTmemCols>(tmem_base);
    }
  }
}

struct DeviceState {
  bool consts = false;
  uint32_t* crc_tables = nullptr;
  int sm_count = 0;
  bool attr[4][2] = {};
};
DeviceState g_dev[16];
std::mutex g_mu;

template <int ALGO, bool SEG>
cudaError_t launch_t(DeviceState& ds, const Params& p, int grid, cudaStream_t st) {
  if (!ds.attr[ALGO][SEG]) {
    cudaError_t e = cudaFuncSetAttribute(bb_xfer_kernel<ALGO, SEG>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(sizeof(SmemT<ALGO>)));
    if (e != cudaSuccess) return e;
    ds.attr[ALGO][SEG] = true;
  }
  bb_xfer_kernel<ALGO, SEG><<<grid, kThreads, sizeof(SmemT<ALGO>), st>>>(p);
  return cudaGetLastError();
}

template <bool SEG>
cudaError_t launch_algo(DeviceState& ds, int algo, const Params& p, int grid, cudaStream_t st) {
  switch (algo) {
    case ALGO_NONE: return launch_t<ALGO_NONE, SEG>(ds, p, grid, st);
    case ALGO_CRC32C: return launch_t<ALGO_CRC32C, SEG>(ds, p, grid, st);
    case ALGO_BBH64: return launch_t<ALGO_BBH64, SEG>(ds, p, grid, st);
    case ALGO_XXH3: return launch_t<ALGO_XXH3, SEG>(ds, p, grid, st);
    default: return cudaErrorNotSupported;
  }
}

}  // namespace

int xfer_smem_bytes(int algo) {
  switch (algo) {
    case ALGO_NONE: return static_cast<int>(sizeof(SmemT<ALGO_NONE>));
    case ALGO_CRC32C: return static_cast<int>(sizeof(SmemT<ALGO_CRC32C>));
    case ALGO_XXH3: return static_cast<int>(sizeof(SmemT<ALGO_XXH3>));
    default: return static_cast<int>(sizeof(SmemT<ALGO_BBH64>));
  }
}

uint32_t crc_unpad_for(uint64_t nbytes) {
  // x^(-8*pad) mod P where pad = zero bytes appended to reach a whole number of tiles.
  // Memoised per pad value (pad < 16384): batches of equal-size objects pay one table hit.
  const uint32_t pad = static_cast<uint32_t>((kTileBytes - (nbytes % kTileBytes)) % kTileBytes);
  static std::mutex mu;
  static std::vector<uint32_t> cache(kTileBytes, 0);  // 0 is never a valid power of x
  {
    std::lock_guard<std::mutex> lk(mu);
    if (cache[pad]) return cache[pad];
  }
  // x^-1 in reflected form: reverse one LFSR bit-step.  Forward: v -> (v>>1) ^ (v&1 ? P : 0);
  // a set top bit means the step XORed P in, so v_prev = ((v ^ P) << 1) | 1.
  static const uint32_t xinv8 = [] {
    uint32_t v = 0x80000000u;  // 1
    for (int i = 0; i < 8; ++i) v = (v & 0x80000000u) ? (((v ^ 0x82F63B78u) << 1) | 1u) : (v << 1);
    return v;  // x^-8
  }();
  uint32_t result = 0x80000000u, base = xinv8;
  for (uint32_t e = pad; e; e >>= 1) {
    if (e & 1) result = gf2_mulmod(result, base);
    base = gf2_mulmod(base, base);
  }
  std::lock_guard<std::mutex> lk(mu);
  cache[pad] = result;
  return result;
}

uint32_t crc_init_term_for(uint64_t nbytes) {
  static std::mutex mu;
  static std::unordered_map<uint64_t, uint32_t> cache;
  {
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(nbytes);
    if (it != cache.end()) return it->second;
  }
  const uint32_t v = gf2_mulmod(0xFFFFFFFFu, gf2_xpow_bytes(nbytes));
  std::lock_guard<std::mutex> lk(mu);
  if (cache.size() > 65536) cache.clear();
  cache.emplace(nbytes, v);
  return v;
}

int launch_xfer(const XferLaunch& l) {
  if (l.ndesc == 0 || l.total_tiles == 0) return 0;
  if (l.small_path && !l.segmented && !l.debug_d && !l.trace_d) return launch_xfer_small(l);
  if (l.segmented && (!l.descs || !l.tile_start)) return static_cast<int>(cudaErrorInvalidValue);
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return static_cast<int>(e);
  if (dev < 0 || dev >= 16) return static_cast<int>(cudaErrorInvalidDevice);
  DeviceState& ds = g_dev[dev];
  {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!ds.consts) {
      uint64_t h[tchash::kN];
      for (uint32_t n = 0; n < tchash::kN; ++n) h[n] = tchash::col_mul(n);
      e = cudaMemcpyToSymbol(c_col_mul, h, sizeof h);
      if (e != cudaSuccess) return static_cast<int>(e);
      uint32_t xp[32];
      uint32_t b = gf2_xpow_bytes(kTileBytes);
      for (int j = 0; j < 32; ++j) {
        xp[j] = b;
        b = gf2_mulmod(b, b);
      }
      e = cudaMemcpyToSymbol(c_xpow_tiles, xp, sizeof xp);
      if (e != cudaSuccess) return static_cast<int>(e);
      e = cudaMemcpyToSymbol(c_xxh_secret, xxh3::kSecret, sizeof xxh3::kSecret);
      if (e != cudaSuccess) return static_cast<int>(e);
      int n = 0;
      if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
      ds.sm_count = n;
      ds.consts = true;
    }
    if (l.algo == ALGO_CRC32C && !ds.crc_tables) {
      static uint32_t host_t[kNumCrcTabs][4][256];
      static bool host_init = false;
      if (!host_init) {
        for (int t = 0; t < kNumCrcTabs; ++t) crc32c_shift_table(kCrcTabBytes[t], host_t[t]);
        host_init = true;
      }
      e = cudaMalloc(reinterpret_cast<void**>(&ds.crc_tables), sizeof host_t);
      if (e != cudaSuccess) return static_cast<int>(e);
      e = cudaMemcpy(ds.crc_tables, host_t, sizeof host_t, cudaMemcpyHostToDevice);
      if (e != cudaSuccess) return static_cast<int>(e);
    }
  }
  Params p;
  p.descs = l.descs;
  p.tile_start = l.tile_start;
  p.use_inline = 0;
  if (l.host_descs && l.ndesc <= kInlineDescs && !l.segmented) {
    p.use_inline = 1;
    std::memcpy(p.inl_descs, l.host_descs, l.ndesc * sizeof(XferDesc));
    std::memcpy(p.inl_tile_start, l.host_tile_start, (l.ndesc + 1) * sizeof(uint32_t));
  }
  p.ndesc = l.ndesc;
  p.total_tiles = l.total_tiles;
  p.sum_ws = reinterpret_cast<unsigned long long*>(l.sum_ws);
  p.done_ws = l.done_ws;
  p.digest_out = l.digest_out;
  p.status_out = l.status_out;
  p.crc_tables = ds.crc_tables;
  p.debug_d = l.debug_d;
  p.trace_d = reinterpret_cast<unsigned long long*>(l.trace_d);
  // Measured on B200 (profiles/xfer_single_gpu.md): 96-128 persistent CTAs saturate HBM for
  // large batches (3.2 TB/s payload); all 148 lose ~6% to DRAM contention.  BB_XFER_CTAS overrides.
  static const int env_ctas = [] { const char* e = std::getenv("BB_XFER_CTAS"); return e ? std::atoi(e) : 0; }();
  // The fused CRC32C is bound by shared-memory lookups per SM, not by DRAM: it takes every SM.
  int grid = l.max_ctas > 0 ? l.max_ctas : env_ctas > 0 ? env_ctas : l.algo == ALGO_CRC32C ? ds.sm_count : std::min(ds.sm_count, 128);
  grid = static_cast<int>(std::min<uint32_t>(static_cast<uint32_t>(grid), l.total_tiles));
  cudaStream_t st = static_cast<cudaStream_t>(l.stream);
  e = l.segmented ? launch_algo<true>(ds, l.algo, p, grid, st) : launch_algo<false>(ds, l.algo, p, grid, st);
  return static_cast<int>(e);
}

}  // namespace bb::gpu
