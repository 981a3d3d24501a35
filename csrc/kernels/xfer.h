// Host-visible API of the sm_100a data-plane kernels (plain C++; no CUDA types leak out).
//
// These kernels replace the reference's UCX call sites (SURVEY K1-K7): `ucp_put_nbx`
// (blackbird_client.cpp:231-237), `ucp_get_nbx` (:315-327) and the CPU byte compare
// (ucx_client.cpp:277).  One launch moves a whole *batch* of objects described by a device
// descriptor table, fusing the transfer with the checksum (and optional replica fan-out).
#pragma once
#include <cstddef>
#include <cstdint>

namespace bb::gpu {

constexpr uint32_t kTileBytes = 16384;   // one TMA tile == one BBH64 tile (tchash_def.h)
constexpr uint32_t kMaxDst = 3;          // replicas written by a single tile pass

enum XferFlags : uint32_t {
  XFER_VERIFY = 1u << 0,    // compare digest with `expect`; status[i] = 1 on mismatch
  XFER_MULTIMEM = 1u << 1,  // dst[0] is an NVLS multicast address: store with multimem.st
  // BBH64 / XXH3 (the tile-sum digests): digest_out receives the *unfinalised* 64-bit tile sum and `reserved` is added to every tile
  // index, so a byte range can be hashed as a slice of a larger object (its sums add up with the slices
  // hashed elsewhere; the host finalises).  With ndst == 0 the descriptor is hash-only (nothing is stored).
  XFER_RAW_SUM = 1u << 2,
  // Segmented objects: the descriptor's bytes come from (GATHER) or go to (SCATTER) a list of device segments instead of
  // one contiguous buffer.  GATHER: `src` points to a segment table.  SCATTER: `dst[0]` points to one (ndst == 1, not
  // with XFER_MULTIMEM).  Digests are those of the concatenated bytes.  Launches that carry either flag must set
  // XferLaunch::segmented; they never take the warp-per-object kernel, the mailbox or the inline parameter table.
  XFER_GATHER = 1u << 3,
  XFER_SCATTER = 1u << 4,
};

// Segment table of one segmented descriptor (device memory, 16-byte aligned): entry 0 is a header whose `addr` holds
// the number of segments n and whose `end` is 0; entries 1..n are the segments in order.  `end` is the cumulative byte
// offset inside the descriptor's range, so segment j covers [table[j-1].end, table[j].end) and table[n].end == nbytes.
// Every segment starts 16-byte aligned and is non-empty; every segment but the last has a length that is a multiple
// of 16.  Overlapping scatter destinations get unspecified bytes (never a fault).
struct XferSeg {
  uint64_t addr;
  uint64_t end;
};
static_assert(sizeof(XferSeg) == 16);

// 64-byte transfer descriptor, one per (object shard, direction).
struct XferDesc {
  const void* src;          // 16-byte aligned; local or peer-mapped
  void* dst[kMaxDst];       // 16-byte aligned; local, peer-mapped or multicast
  uint64_t nbytes;
  uint32_t first_tile;      // exclusive prefix sum of ceil(nbytes / kTileBytes)
  uint32_t ndst;
  uint64_t expect;          // BBH64: expected digest.  CRC32C: (init_term << 32) | expected crc
  uint32_t flags;
  uint32_t reserved;        // CRC32C: x^(-8*pad) mod P (crc_unpad_for); BBH64 + XFER_RAW_SUM: tile index base
};
static_assert(sizeof(XferDesc) == 64, "XferDesc must be 64 bytes");

constexpr uint32_t kSmallBytes = 4096;     // objects up to this size may take the warp-per-object path (xfer_small.cu)
constexpr uint32_t kSmallPending = 0xFFFFFFFFu;  // value of a status slot whose object has not completed yet (flag completion)
constexpr uint32_t kInlineDescs = 8;       // descriptors that fit in the kernel parameter block
constexpr uint32_t kDirectResults = 64;    // batches up to this size write digests straight to pinned host memory

enum XferAlgo : int { ALGO_NONE = 0, ALGO_CRC32C = 1, ALGO_BBH64 = 2, ALGO_XXH3 = 3 };

struct XferLaunch {
  const XferDesc* descs = nullptr;       // device pointer, ndesc entries
  const uint32_t* tile_start = nullptr;  // device pointer, ndesc+1 entries (prefix sums)
  uint32_t ndesc = 0;
  uint32_t total_tiles = 0;
  uint64_t* sum_ws = nullptr;            // device, ndesc entries, must be zero on entry (self-cleaning)
  uint32_t* done_ws = nullptr;           // device, ndesc entries, must be zero on entry (self-cleaning)
  uint64_t* digest_out = nullptr;        // device, ndesc entries
  uint32_t* status_out = nullptr;        // device, ndesc entries (0 ok / 1 checksum mismatch)
  const uint32_t* crc_tables = nullptr;  // device, CRC32C shift tables (only ALGO_CRC32C)
  uint32_t* debug_d = nullptr;           // optional: raw accumulators [tile][128][16] (tests)
  uint64_t* trace_d = nullptr;           // optional: per-tile pipeline timestamps [tile][4] (globaltimer ns)
  // Optional host copies of the two tables: batches of <= kInlineDescs descriptors travel in the
  // kernel parameters instead (descs / tile_start may then be null).
  const XferDesc* host_descs = nullptr;
  const uint32_t* host_tile_start = nullptr;
  int algo = ALGO_BBH64;
  bool small_path = false;               // every descriptor is <= kSmallBytes, none is a RAW_SUM slice: warp-per-object kernel
  bool flag_completion = false;          // small path only: status_out (pinned, preset to kSmallPending) is the completion flag
  bool segmented = false;                // some descriptor carries XFER_GATHER / XFER_SCATTER: device tables only
  int max_ctas = 0;                      // 0 = one CTA per SM
  void* stream = nullptr;                // cudaStream_t
};

// Returns 0 on success, else a cudaError_t value.
int launch_xfer(const XferLaunch& l);
// ---- mailbox (xfer_small.cu): a resident warp fed through pinned host memory, so that a single small put / get costs no
// kernel launch.  All three structures live in pinned host memory (the device reads / writes them over PCIe).
constexpr uint32_t kMailSlots = 16;
struct MailSlot {  // 64 bytes = one cache line = one PCIe read; the host writes `seq` LAST
  uint64_t src;
  uint64_t dst;
  uint64_t expect;     // as XferDesc::expect
  uint32_t nbytes;     // <= kSmallBytes
  uint32_t flags;      // XferFlags (no MULTIMEM, no RAW_SUM)
  uint32_t algo;       // XferAlgo
  uint32_t reserved;   // as XferDesc::reserved
  uint32_t pad[5];
  uint32_t seq;        // word 15
};
static_assert(sizeof(MailSlot) == 64, "MailSlot must be one cache line");
struct alignas(64) MailResult {  // 64 bytes; the device writes the first 16 bytes (digest, status, seq) with one store
  uint64_t digest;
  uint32_t status;
  uint32_t seq;
  uint32_t pad[12];
};
static_assert(sizeof(MailResult) == 64 && offsetof(MailResult, seq) == 12);
struct MailCtl {
  uint32_t exit_epoch;  // epoch of the last kernel incarnation that has exited (== the launched epoch: nobody is polling)
  uint32_t next_seq;    // first sequence number that incarnation did NOT consume
  uint32_t pad[14];
};
// Launches one incarnation of the mailbox kernel on `stream`: it serves requests from sequence number `first_seq` on and
// exits after `linger_ns` without a request or `max_ns` in total, then writes (next_seq, exit_epoch = epoch) into *ctl.
int launch_mailbox(const MailSlot* slots, MailResult* results, MailCtl* ctl, uint32_t first_seq, uint32_t epoch, uint64_t linger_ns,
                   uint64_t max_ns, void* stream);

// Small-object latency tier: one warp per descriptor, digest bit-identical to launch_xfer's (needs descs; not tile_start).
int launch_xfer_small(const XferLaunch& l);
int xfer_smem_bytes(int algo);
// Fused MXFP8 transfer (xfer_mxfp8.cu).  The packed object is one contiguous [payload n][scales n/32] extent.
// Descriptors: pack (put): src = bf16 source, dst[0..ndst-1] = base of the packed object in every replica (the scales
// follow the payload), nbytes = payload bytes (= elements, a multiple of kTileBytes); unpack (get): src = base of the
// packed object, dst[0] = bf16 destination.  `sum_ws` receives the unfinalised
// BBH64 sum of the payload tiles per descriptor (must be zero on entry); descs / tile_start are device tables.
int launch_xfer_fp8(const XferLaunch& l, bool unpack);
int xfer_fp8_smem_bytes();

// CRC32C per-object constants (host): un-padding multiplier and the init-register term.
uint32_t crc_unpad_for(uint64_t nbytes);
uint32_t crc_init_term_for(uint64_t nbytes);

// Number of tiles of an object (0 for empty objects).
inline uint32_t tiles_of(uint64_t nbytes) { return static_cast<uint32_t>((nbytes + kTileBytes - 1) / kTileBytes); }

// ---- comparators / utilities (baseline.cu)
// Plain vectorised copy kernel (the "unfused copy kernel" comparator of BASELINE.md §4).
int launch_copy_simt(void* dst, const void* src, uint64_t nbytes, void* stream);
// Stand-alone CRC32C over device memory (comparator: "separate CRC32C kernel"); result is the
// standard CRC32C written to *out (device).  `tables` = device copy of crc tables (see crc_tables_host()).
int launch_crc32c_simt(const void* data, uint64_t nbytes, uint32_t* out, uint32_t* scratch, void* stream);
// L2 flush helper: writes `nbytes` of a scratch buffer.
int launch_fill(void* dst, uint64_t nbytes, uint32_t value, void* stream);
// Fills a buffer with deterministic pseudo-random bytes (synthetic objects).
int launch_random_fill(void* dst, uint64_t nbytes, uint64_t seed, void* stream);

// MXFP8 pack / unpack (mxfp8.cu): bf16 <-> [E4M3 payload | E8M0 scale per 32 elements].
// n_elems % 32 == 0; packed size = n_elems + n_elems / 32 bytes (common/mxfp8.h).
int launch_mxfp8_pack(const void* src_bf16, uint64_t n_elems, void* dst_packed, void* stream);
int launch_mxfp8_unpack(const void* src_packed, uint64_t n_elems, void* dst_bf16, void* stream);

}  // namespace bb::gpu
