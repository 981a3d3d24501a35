// BlackbirdClient: the SDK (SURVEY C19).
//
// Parity: reference include/blackbird/client/blackbird_client.h:22-139 — BlackbirdClientOptions
// (keystone_host/port, rpc_timeout, io_parallelism), connect, object_exists, get_workers,
// get(key) -> bytes, put(key, ptr, size, cfg), put(key, vector, cfg), remove.
// New surface required by BASELINE.json: batch_put / batch_get for host buffers and for device
// pointers (the fused NVLink kernel path, installed by fabric/gpu_fabric.h as a DeviceTransport).
//
// Behavioural fixes over the reference: rpc_timeout and io_parallelism are honoured (:204-205
// ignores them); the source pointer of a shard is `data + running offset` (not `data +
// remote_addr`, bug #8); connections to workers are cached instead of re-created per call;
// every shard is checksummed and verified; reads fail over to the next replica; a failed put is
// cancelled.
#pragma once
#include <atomic>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "common/metrics.h"
#include "net/tcp.h"
#include "rpc/rpc_service.h"

namespace bb::client {

struct BlackbirdClientOptions {
  std::string keystone_host = "127.0.0.1";
  uint16_t keystone_port = 9090;
  // HA deployments: every keystone ("host:port"); when set it replaces keystone_host/port and the control connection
  // follows the elected leader (KeystoneRpcClient::connect_any).
  std::vector<std::string> keystone_endpoints;
  int rpc_timeout_ms = 30000;
  size_t io_parallelism = 4;
  std::string node_id;        // where this client runs (locality-aware placement)
  bool register_session = false;
  // Same-host fast path: DRAM pools that their worker backs with a memfd (`shared_memory: true`) are mapped into this
  // process and shards are moved with memcpy instead of the TCP data server (the role UCX's shared-memory transports
  // play for the reference's intra-node RMA).  BB_DISABLE_SHM=1 in the environment also turns it off.
  bool enable_shm = true;
  std::string auth_token;  // shared cluster token (net/tcp.h); empty = BB_AUTH_TOKEN / open cluster
  bool encrypt_transport = false;  // secure mode of the RPC protocol (net/tcp.h); also BB_ENCRYPT_TRANSPORT=1
  std::string auth_token_ro;       // read-only membership: set this INSTEAD of auth_token (net/tcp.h); also BB_AUTH_TOKEN_RO
  // Tenant identity (common/tenant.h): set these INSTEAD of a member token.  The servers then know who is calling: keys
  // outside the tenant's grants are ACCESS_DENIED, puts beyond its budget QUOTA_EXCEEDED.  Also BB_TENANT / BB_TENANT_SECRET.
  std::string tenant, tenant_secret;
};

// One device-side transfer request of a batch (a shard).
struct DeviceShardOp {
  size_t item = 0;            // index of the object in the batch
  size_t copy = 0, shard = 0;
  const ShardPlacement* placement = nullptr;
  std::vector<const ShardPlacement*> replicas;  // same shard on the other copies (put fan-out)
  uint64_t obj_offset = 0;    // byte offset of this shard inside the object
  // Segmented object (gather put / scatter get): the object's whole segment list, or null for a contiguous object at
  // dev_ptrs[item].  The transport moves the slice [obj_offset, obj_offset + placement->length) of it.
  const DeviceSegment* segs = nullptr;
  size_t nsegs = 0;
};

// Finds the slice [offset, offset + length) of a segment list: index of its first segment and the bytes of that segment
// before the slice (the slice runs on through the following segments).  Returns false when the list is too short.
inline bool segment_slice(const DeviceSegment* segs, size_t nsegs, uint64_t offset, size_t* first, uint64_t* skip) {
  uint64_t pos = 0;
  for (size_t k = 0; k < nsegs; pos += segs[k].len, ++k)
    if (offset < pos + segs[k].len) {
      *first = k;
      *skip = offset - pos;
      return true;
    }
  return false;
}

// One object of a fused MXFP8 transfer: the whole packed object ([E4M3 payload][E8M0 scales]) is a single shard.
struct DeviceFp8Op {
  const ShardPlacement* placement = nullptr;
  void* wide = nullptr;     // client's bf16 tensor (source of a put, destination of a get)
  uint64_t n_elems = 0;
  std::vector<const ShardPlacement*> replicas;  // put: the other copies (<= 2), written by the same tile pass
};

// Implemented by the GPU fabric: moves shards between client device buffers and worker slabs
// with the fused kernels.  Returns per-op digests (put) or verifies them (get).
class DeviceTransport {
 public:
  virtual ~DeviceTransport() = default;
  // dev_ptrs[item] is the client's device buffer of object `item`.
  virtual ErrorCode put_shards(const std::vector<DeviceShardOp>& ops, const std::vector<const void*>& dev_ptrs,
                               ChecksumAlgo algo, void* stream, std::vector<uint64_t>* digests) = 0;
  virtual ErrorCode get_shards(const std::vector<DeviceShardOp>& ops, const std::vector<void*>& dev_ptrs, ChecksumAlgo algo,
                               void* stream, std::vector<uint32_t>* status) = 0;
  virtual bool can_reach(const ShardPlacement& s) const = 0;
  virtual uint64_t launches() const = 0;
  // Asynchronous variants: enqueue the fused launch and return a ticket, so the caller can overlap
  // control-plane round trips of the next chunk with this chunk's transfer.  Default = synchronous.
  virtual Result<uint64_t> submit_put(const std::vector<DeviceShardOp>& ops, const std::vector<const void*>& dev_ptrs, ChecksumAlgo algo,
                                      void* stream) {
    std::vector<uint64_t> d;
    ErrorCode ec = put_shards(ops, dev_ptrs, algo, stream, &d);
    if (ec != ErrorCode::OK) return ec;
    sync_results_[++sync_ticket_] = {std::move(d), {}};
    return sync_ticket_;
  }
  virtual ErrorCode wait_put(uint64_t ticket, std::vector<uint64_t>* digests) {
    auto it = sync_results_.find(ticket);
    if (it == sync_results_.end()) return ErrorCode::NOT_FOUND;
    if (digests) *digests = std::move(it->second.first);
    sync_results_.erase(it);
    return ErrorCode::OK;
  }
  virtual Result<uint64_t> submit_get(const std::vector<DeviceShardOp>& ops, const std::vector<void*>& dev_ptrs, void* stream) {
    std::vector<uint32_t> st;
    ErrorCode ec = get_shards(ops, dev_ptrs, ChecksumAlgo::NONE, stream, &st);
    if (ec != ErrorCode::OK) return ec;
    sync_results_[++sync_ticket_] = {{}, std::move(st)};
    return sync_ticket_;
  }
  virtual ErrorCode wait_get(uint64_t ticket, std::vector<uint32_t>* status) {
    auto it = sync_results_.find(ticket);
    if (it == sync_results_.end()) return ErrorCode::NOT_FOUND;
    if (status) *status = std::move(it->second.second);
    sync_results_.erase(it);
    return ErrorCode::OK;
  }
  // True when the shard lives in this client's own device memory (a get from it never leaves the GPU).
  virtual bool is_local(const ShardPlacement& s) const { return false; }
  virtual size_t max_in_flight() const { return 1; }
  // Fused MXFP8 put / get (pack / unpack inside the transfer kernel).  digests[i] = BBH64 of the stored packed
  // object; status[i] != 0 = digest mismatch on get.  Objects must satisfy fp8_eligible().
  // Prometheus lines of the transport's own counters (bytes per path, launches, ...); appended to the client's metrics.
  virtual std::string metrics_text() const { return {}; }
  virtual bool fp8_eligible(uint64_t n_elems) const { return false; }
  virtual ErrorCode put_fp8(const std::vector<DeviceFp8Op>& ops, void* stream, std::vector<uint64_t>* digests) { return ErrorCode::NOT_IMPLEMENTED; }
  virtual ErrorCode get_fp8(const std::vector<DeviceFp8Op>& ops, void* stream, std::vector<uint32_t>* status) { return ErrorCode::NOT_IMPLEMENTED; }
  // Staging copies for objects (or shards) that live on host tiers: device <-> host buffer, synchronous.
  virtual ErrorCode copy_h2d(void* dev, const void* host, size_t n, void* stream) { return ErrorCode::NOT_IMPLEMENTED; }
  virtual ErrorCode copy_d2h(void* host, const void* dev, size_t n, void* stream) { return ErrorCode::NOT_IMPLEMENTED; }

 private:
  uint64_t sync_ticket_ = 0;
  std::map<uint64_t, std::pair<std::vector<uint64_t>, std::vector<uint32_t>>> sync_results_;
};

class HostLoopbackTransport;

class BlackbirdClient {
 public:
  explicit BlackbirdClient(BlackbirdClientOptions opts = {});
  // In-process deployment: talk to a KeystoneApi directly (no TCP to the control plane).
  BlackbirdClient(std::shared_ptr<rpc::KeystoneApi> keystone, BlackbirdClientOptions opts = {});
  ~BlackbirdClient();

  ErrorCode connect();
  bool connected() const { return keystone_ != nullptr; }
  const std::string& session_id() const { return session_id_; }

  // ---- reference API
  Result<bool> object_exists(const ObjectKey& key);
  Result<std::vector<CopyPlacement>> get_workers(const ObjectKey& key);
  Result<std::vector<uint8_t>> get(const ObjectKey& key);
  ErrorCode get_into(const ObjectKey& key, void* buf, size_t capacity, size_t* out_size);
  ErrorCode put(const ObjectKey& key, const uint8_t* data, size_t size, const WorkerConfig& cfg = {});
  ErrorCode put(const ObjectKey& key, const std::vector<uint8_t>& data, const WorkerConfig& cfg = {}) {
    return put(key, data.data(), data.size(), cfg);
  }
  ErrorCode remove(const ObjectKey& key);
  // bf16 tensors stored as MXFP8 (common/mxfp8.h layout) with the pack fused into the put kernel and the unpack
  // into the get kernel.  n_elems[i] must be a multiple of 32 (whole MX blocks; pad + mxfp8_pack otherwise); up to 3 copies
  // (written by one tile pass: converted once, stored to every replica; gets fail over between them), one
  // shard per object.  The stored object is identical to packing first and putting the packed bytes.
  std::vector<ErrorCode> batch_put_device_fp8(const std::vector<ObjectKey>& keys, const std::vector<const void*>& bf16_ptrs,
                                              const std::vector<uint64_t>& n_elems, const WorkerConfig& cfg, void* stream);
  std::vector<ErrorCode> batch_get_device_fp8(const std::vector<ObjectKey>& keys, const std::vector<void*>& bf16_ptrs,
                                              const std::vector<uint64_t>& n_elems, void* stream);
  bool device_fp8_eligible(uint64_t n_elems) const { return device_ && device_->fp8_eligible(n_elems); }
  // Moves every copy of the object to `target` (promotion to the GPU tier, demotion to DRAM / NVMe ...).
  ErrorCode migrate(const ObjectKey& key, StorageClass target);

  // ---- batched host-memory API
  std::vector<ErrorCode> batch_put(const std::vector<ObjectKey>& keys, const std::vector<const uint8_t*>& data,
                                   const std::vector<size_t>& sizes, const WorkerConfig& cfg = {});
  std::vector<Result<std::vector<uint8_t>>> batch_get(const std::vector<ObjectKey>& keys);
  std::vector<ErrorCode> batch_remove(const std::vector<ObjectKey>& keys);
  std::vector<Result<bool>> batch_exists(const std::vector<ObjectKey>& keys);

  // ---- batched device-memory API (fused kernels; requires a DeviceTransport)
  void set_device_transport(std::shared_ptr<DeviceTransport> t) { device_ = std::move(t); }
  std::vector<ErrorCode> batch_put_device(const std::vector<ObjectKey>& keys, const std::vector<const void*>& dev_ptrs,
                                          const std::vector<size_t>& sizes, const WorkerConfig& cfg, void* stream);
  // out_sizes[i] receives the object size; buffers must be large enough (capacity[i]).
  std::vector<ErrorCode> batch_get_device(const std::vector<ObjectKey>& keys, const std::vector<void*>& dev_ptrs,
                                          const std::vector<size_t>& capacity, void* stream, std::vector<size_t>* out_sizes);
  // Segmented objects (a paged KV cache: one object = many blocks spread over many tensors).  Object i is the
  // concatenation of the next seg_counts[i] entries of `segs`; it is stored exactly as a contiguous put of that
  // concatenation would store it (same bytes, same digests), so every other read / write path works on it.
  // Each segment: ptr 16-byte aligned, len > 0, len % 16 == 0 except for the object's last segment; at most
  // kMaxObjectSegments segments per object.  An object breaking these rules is INVALID_PARAMETERS (VALUE_OUT_OF_RANGE
  // for too many segments) and the rest of the batch proceeds; seg_counts that do not add up to segs.size() make the
  // whole batch INVALID_PARAMETERS.  Get: the stored size must equal the sum of the segment lengths (else
  // INVALID_PARAMETERS, nothing written).  Overlapping scatter destinations receive unspecified bytes.
  static constexpr size_t kMaxObjectSegments = size_t{1} << 20;
  std::vector<ErrorCode> batch_put_device_gather(const std::vector<ObjectKey>& keys, const std::vector<DeviceSegment>& segs,
                                                 const std::vector<uint32_t>& seg_counts, const WorkerConfig& cfg, void* stream);
  std::vector<ErrorCode> batch_get_device_scatter(const std::vector<ObjectKey>& keys, const std::vector<DeviceSegment>& segs,
                                                  const std::vector<uint32_t>& seg_counts, void* stream);

  Result<ClusterStats> cluster_stats();
  rpc::KeystoneApi& keystone() { return *keystone_; }
  std::string metrics_text() const { return metrics_.render("bb_client_") + (device_ ? device_->metrics_text() : std::string()); }
  // Device batches are split into `chunks` pipelined launches; 0 = decide from the measured RPC latency.
  void set_device_pipeline_chunks(size_t chunks) { pipeline_chunks_ = chunks; }
  std::map<std::string, std::vector<double>> phase_summary() const { return metrics_.histogram_summary(); }

 private:
  friend class HostLoopbackTransport;
  struct WorkerConn;
  std::shared_ptr<net::RpcClient> acquire(const std::string& endpoint);
  void release(const std::string& endpoint, std::shared_ptr<net::RpcClient> c);
  ErrorCode write_shard(const ShardPlacement& s, const uint8_t* src, uint64_t* digest, ChecksumAlgo algo);
  ErrorCode read_shard(const ShardPlacement& s, uint8_t* dst, ChecksumAlgo algo);
  ErrorCode put_once(const ObjectKey& key, const uint8_t* data, size_t size, const WorkerConfig& cfg);
  ErrorCode transfer_put(const std::vector<CopyPlacement>& copies, const uint8_t* data, ChecksumAlgo algo,
                         keystone::ShardChecksums* sums);
  ErrorCode transfer_get(const std::vector<CopyPlacement>& copies, uint8_t* dst, size_t size);
  ErrorCode get_with_refresh(const ObjectKey& key, uint8_t* (*alloc)(void*, size_t), void* ctx, size_t capacity, size_t* out_size);
  static uint64_t shard_offset(const ShardPlacement& s);
  static ChecksumAlgo algo_of(const std::vector<CopyPlacement>& copies, ChecksumAlgo hint);
  // [begin, end) index ranges that split a batch so that transfers of one chunk overlap the
  // control-plane round trips of its neighbours (large batches only).
  std::vector<std::pair<size_t, size_t>> plan_chunks(const std::vector<size_t>& sizes, double rpc_us_per_object) const;
  // Segment lists of a segmented batch: object i is segs[first[i] .. first[i] + count[i]).
  struct SegView {
    const DeviceSegment* segs = nullptr;
    std::vector<size_t> first, count;
  };
  // Bodies of batch_{put,get}_device and of their segmented variants (`sv` null = contiguous objects at dev_ptrs).
  std::vector<ErrorCode> put_device_impl(const std::vector<ObjectKey>& keys, const std::vector<const void*>& dev_ptrs,
                                         const std::vector<size_t>& sizes, const SegView* sv, const WorkerConfig& cfg, void* stream);
  std::vector<ErrorCode> get_device_impl(const std::vector<ObjectKey>& keys, const std::vector<void*>& dev_ptrs,
                                         const std::vector<size_t>& capacity, const SegView* sv, void* stream,
                                         std::vector<size_t>* out_sizes);

  // Mapped shared DRAM pools (same-host fast path); a mapping is dropped when the pool re-registers under a new key.
  struct ShmPool {
    uint8_t* base = nullptr;
    uint64_t size = 0;
    uint64_t remote_base = 0;
    std::vector<uint8_t> key;
  };
  uint8_t* shm_resolve(const ShardPlacement& s);
  std::mutex shm_mu_;
  std::map<std::string, ShmPool> shm_pools_;
  std::map<std::string, std::vector<uint8_t>> shm_unreachable_;  // pool -> key that could not be mapped

  BlackbirdClientOptions opts_;
  std::shared_ptr<rpc::KeystoneApi> keystone_;
  std::shared_ptr<DeviceTransport> device_;
  size_t pipeline_chunks_ = 0;  // 0 = adaptive (from the measured control-plane latency)
  std::atomic<double> put_rpc_us_per_obj_{0}, get_rpc_us_per_obj_{0};
  std::string session_id_;
  std::mutex conn_mu_;
  std::map<std::string, std::vector<std::shared_ptr<net::RpcClient>>> idle_conns_;
  mutable Metrics metrics_;
};

// A DeviceTransport without a GPU: "device pointers" are host pointers and shards move over the host data paths of a
// second (I/O) client.  It exists so that the device-side client logic -- chunk planning and pipelining, fan-out
// descriptors, replica choice and fail-over, host-staged fall-backs, placement refresh -- is testable on CPU-only
// machines (the reference has no fake transport at all, SURVEY section 4); the GPU fabric replaces it in production.
class HostLoopbackTransport : public DeviceTransport {
 public:
  // `io` moves the bytes (its own connections / shared-memory mappings); it must outlive the transport.
  explicit HostLoopbackTransport(std::shared_ptr<BlackbirdClient> io, bool reach_disk_tiers = false)
      : io_(std::move(io)), reach_disk_(reach_disk_tiers) {}
  ErrorCode put_shards(const std::vector<DeviceShardOp>& ops, const std::vector<const void*>& dev_ptrs, ChecksumAlgo algo, void* stream,
                       std::vector<uint64_t>* digests) override;
  ErrorCode get_shards(const std::vector<DeviceShardOp>& ops, const std::vector<void*>& dev_ptrs, ChecksumAlgo algo, void* stream,
                       std::vector<uint32_t>* status) override;
  bool can_reach(const ShardPlacement& s) const override;
  uint64_t launches() const override { return launches_; }
  ErrorCode copy_h2d(void* dev, const void* host, size_t n, void*) override {
    std::memcpy(dev, host, n);
    return ErrorCode::OK;
  }
  ErrorCode copy_d2h(void* host, const void* dev, size_t n, void*) override {
    std::memcpy(host, dev, n);
    return ErrorCode::OK;
  }
  size_t max_in_flight() const override { return 2; }
  // MXFP8 through the CPU reference codec (common/mxfp8.h): the stored object and its digest are the ones the fused
  // kernels produce, so the fp8 client logic (replica fan-out, fail-over between replicas) is testable on CPU too.
  bool fp8_eligible(uint64_t n_elems) const override { return n_elems != 0 && n_elems % 32 == 0; }
  ErrorCode put_fp8(const std::vector<DeviceFp8Op>& ops, void* stream, std::vector<uint64_t>* digests) override;
  ErrorCode get_fp8(const std::vector<DeviceFp8Op>& ops, void* stream, std::vector<uint32_t>* status) override;

 private:
  // Segmented op: copies the shard's slice of the segment list into (gather) or out of (scatter) `buf`.
  static ErrorCode copy_segments(const DeviceShardOp& op, uint8_t* buf, bool gather);
  std::shared_ptr<BlackbirdClient> io_;
  bool reach_disk_;
  std::atomic<uint64_t> launches_{0};
};

}  // namespace bb::client
