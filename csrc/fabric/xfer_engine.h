// XferEngine: host-side driver of the fused transfer kernel.
//
// Owns per-device descriptor rings (pinned host staging + device tables + self-cleaning digest
// workspace) so that a batched put/get costs: one small H2D copy of the descriptor table, ONE
// kernel launch, one small D2H copy of digests/status.  This is what replaces the reference
// client's per-shard `UcxContext` + endpoint create/destroy + `ucp_put_nbx` + busy-poll
// (blackbird_client.cpp:204-274, 276-351): zero per-object setup, zero per-object launches.
#pragma once
#include <cstdint>
#include <memory>
#include <vector>

#include "common/checksum.h"
#include "common/error.h"
#include "common/result.h"
#include "common/types.h"
#include "kernels/xfer.h"

namespace bb::gpu {

// One piece of a segmented item (common/types.h).
using XferSegment = DeviceSegment;

// Segment table entries one launch may carry (segments plus one header per segmented item, kernels/xfer.h XferSeg).
constexpr uint64_t kMaxSegTableEntries = 1ull << 21;

struct XferItem {
  const void* src = nullptr;
  void* dst[kMaxDst] = {nullptr, nullptr, nullptr};
  uint32_t ndst = 1;
  uint64_t nbytes = 0;
  uint64_t expect = 0;   // expected digest when flags & XFER_VERIFY
  uint32_t flags = 0;
  uint32_t tile_base = 0;  // XFER_RAW_SUM: index of this slice's first tile inside the hashed object
  // Segmented source (flags & XFER_GATHER, replaces `src`) or destination (flags & XFER_SCATTER, replaces `dst[0]`;
  // ndst == 1): the item's bytes are segs[0..nsegs) with the first `seg_skip` bytes of segs[0] left out, cut at
  // `nbytes`.  The list must cover nbytes; every piece must start 16-byte aligned and every piece but the last must be a
  // multiple of 16 bytes long.  submit() packs the tables after the descriptor table (same H2D copy).
  const XferSegment* segs = nullptr;
  uint32_t nsegs = 0;
  uint64_t seg_skip = 0;
};

// One object of a fused MXFP8 transfer: `wide` is the caller's bf16 tensor, `packed` the slab location of the
// stored object ([E4M3 payload n_elems][E8M0 scales n_elems / 32]).
struct Fp8Item {
  void* wide = nullptr;
  void* packed = nullptr;            // replica 0 (the copy a get reads)
  void* more_packed[kMaxDst - 1] = {nullptr, nullptr};  // put: further replicas written by the same tile pass
  uint32_t nreplicas = 1;            // put: 1..kMaxDst
  uint64_t n_elems = 0;   // multiple of 32 (whole MX blocks)
  uint64_t expect = 0;    // unpack + verify: digest recorded at put time
  bool verify = false;
};

struct XferResult {
  std::vector<uint64_t> digest;  // per item
  std::vector<uint32_t> status;  // per item: 0 ok, 1 checksum mismatch
  float device_ms = 0.f;         // kernel time (CUDA events) of the batch
};

class XferEngine {
 public:
  // `device` is the CUDA ordinal the kernels run on; `max_items` bounds one batch.
  static Result<std::unique_ptr<XferEngine>> create(int device, uint32_t max_items = 1u << 16, int slots = 4);
  ~XferEngine();
  XferEngine(const XferEngine&) = delete;
  XferEngine& operator=(const XferEngine&) = delete;

  // Enqueues the whole batch on `stream` (cudaStream_t, nullptr = legacy default stream) and
  // returns a ticket.  Does not block (unless all slots are in flight).
  Result<uint64_t> submit(const std::vector<XferItem>& items, ChecksumAlgo algo, void* stream,
                          bool capture_debug = false);
  // Blocks until the ticket's batch has finished on the device and fills `out`.
  ErrorCode wait(uint64_t ticket, XferResult* out);
  // Convenience: submit + wait.
  ErrorCode run(const std::vector<XferItem>& items, ChecksumAlgo algo, void* stream, XferResult* out);
  // Fused MXFP8 put (pack = bf16 -> slab) or get (unpack = slab -> bf16): the bf16 side is read / written once, the
  // E4M3 payload is hashed on the tensor cores while it sits in shared memory, and the digest returned is the
  // BBH64 of the stored packed object (identical to hashing the output of mxfp8_pack).  Synchronous.
  ErrorCode run_fp8(const std::vector<Fp8Item>& items, bool unpack, void* stream, XferResult* out);
  static bool fp8_eligible(uint64_t n_elems) { return n_elems != 0 && n_elems % 32 == 0; }  // whole MX blocks

  // Raw accumulators of the last capture_debug batch: [total_tiles][128][16] (tests only).
  const std::vector<uint32_t>& debug_accumulators() const { return debug_host_; }
  // Diagnostics: when on, every batch records per-tile pipeline timestamps (globaltimer ns):
  // [tile][4] = load issued, landed in shared memory, store issued, slot released.  Read after wait().
  void set_tile_trace(bool on) { tile_trace_ = on; }
  const std::vector<uint64_t>& tile_trace() const { return trace_host_; }

  int device() const { return device_; }
  uint64_t launches() const { return launches_; }  // kernels launched so far
  uint64_t small_launches() const { return small_launches_; }  // of which warp-per-object launches (xfer_small.cu)
  // Batches made only of objects <= kSmallBytes take the warp-per-object kernel (default on; BB_XFER_SMALL=0 disables).
  void set_small_path(bool on) { small_path_ = on; }
  // Small batches (<= kDirectResults objects on the warp path) complete by a flag in pinned memory instead of CUDA
  // events (default on; BB_XFER_FLAG_COMPLETION=0 disables).  Their XferResult::device_ms is 0 (not measured).
  void set_flag_completion(bool on) { flag_completion_ = on; }
  // Batches of <= 8 single-destination small objects whose stream has nothing pending are handed to the resident mailbox
  // warp (xfer_small.cu) instead of being launched: no cudaLaunchKernel in the steady state.  Default on;
  // BB_XFER_MAILBOX=0 disables; BB_MAILBOX_LINGER_US (default 200) = how long the warp waits for the next request.
  void set_mailbox(bool on) { mailbox_on_ = on; }
  uint64_t mailbox_requests() const { return mailbox_requests_; }   // objects served by the resident warp
  uint64_t mailbox_launches() const { return mailbox_launches_; }   // incarnations of the mailbox kernel
  void set_max_ctas(int n) { max_ctas_ = n; }
  int last_cuda_error() const { return last_cuda_error_; }

 private:
  struct Slot;
  XferEngine() = default;
  int device_ = 0;
  uint32_t max_items_ = 0;
  std::vector<std::unique_ptr<Slot>> slots_;
  uint64_t next_ticket_ = 1;
  uint64_t launches_ = 0;
  uint64_t small_launches_ = 0;
  bool small_path_ = true;
  bool flag_completion_ = true;
  bool mailbox_on_ = true;
  bool mailbox_enabled();
  struct Mailbox;
  std::unique_ptr<Mailbox> mb_;
  ErrorCode mailbox_post(Slot* s, const XferDesc* descs, uint32_t nd, int algo);
  ErrorCode mailbox_wait(Slot* s);
  ErrorCode mailbox_launch_locked(uint32_t first_seq);
  uint64_t mailbox_requests_ = 0, mailbox_launches_ = 0;
  bool small_path_enabled();
  bool flag_completion_enabled();
  int max_ctas_ = 0;
  int last_cuda_error_ = 0;
  std::vector<uint32_t> debug_host_;
  bool tile_trace_ = false;
  std::vector<uint64_t> trace_host_;
  struct Fp8State;
  std::unique_ptr<Fp8State> fp8_;
};

// Device helpers used by bindings, the worker and benchmarks (all return ErrorCode).
ErrorCode device_count(int* n);
ErrorCode device_malloc(int device, uint64_t bytes, void** out);
ErrorCode device_free(int device, void* p);
ErrorCode host_alloc_pinned(uint64_t bytes, void** out);
ErrorCode host_free_pinned(void* p);
ErrorCode stream_synchronize(void* stream);
ErrorCode device_synchronize(int device);
const char* cuda_error_string(int code);
// Comparator helpers (return a cudaError_t value).
int device_memcpy_peer_async(void* dst, int dst_device, const void* src, int src_device, uint64_t nbytes, void* stream);
int device_enable_peer_access(int device, int peer);

}  // namespace bb::gpu
