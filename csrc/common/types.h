// Core value types of the object store.
//
// Parity: reference include/blackbird/common/types.h — ids (:51-65), StorageClass (:82-92),
// placement model UcxEndpoint/MemoryLocation/FileLocation/CxlMemoryLocation/LocationDetail/
// ShardPlacement/CopyPlacement (:97-156), WorkerConfig (:161-187), ClusterStats (:192-209),
// KeystoneConfig (:410-444), ClientConfig (:449-459), MemoryPool (:464-493), hash<UUID> (:499-512).
// B200-native additions: GpuSlabLocation (rank/slab/offset addressing of an exported HBM
// slab — the role the (remote_addr, rkey) pair plays for UCX), per-shard checksum, checksum /
// fp8-pack / NVLS policy knobs, pool topology attributes that the placement engine consumes.
#pragma once
#include <chrono>
#include <cstdint>
#include <optional>
#include <string>
#include <string_view>
#include <utility>
#include <variant>
#include <vector>

#include "common/cxl_config.h"
#include "common/checksum.h"
#include "common/error.h"
#include "common/json.h"
#include "common/result.h"

namespace bb {

using ObjectKey = std::string;

// `len` bytes at device (or device-accessible) address `ptr`: one piece of a segmented object, whose bytes are the
// concatenation of its segments (BlackbirdClient::batch_put_device_gather / batch_get_device_scatter).
struct DeviceSegment {
  uint64_t ptr = 0;
  uint64_t len = 0;
};
using Version = uint64_t;
using MemoryPoolId = std::string;
using NodeId = std::string;
using WorkerId = std::string;
using UUID = std::pair<uint64_t, uint64_t>;
using ViewVersionId = int64_t;
using LeaseId = int64_t;

inline constexpr const char* DEFAULT_CLUSTER_ID = "blackbird_cluster";
inline constexpr double DEFAULT_HIGH_WATERMARK = 0.9;
inline constexpr int64_t DEFAULT_CLIENT_TTL_SEC = 10;
inline constexpr size_t DEFAULT_REPLICATION_FACTOR = 3;
inline constexpr size_t DEFAULT_MAX_WORKERS_PER_COPY = 4;

using Clock = std::chrono::steady_clock;
using TimePoint = Clock::time_point;

// Numeric values match the reference enum (types.h:82-92).
enum class StorageClass : uint32_t {
  STORAGE_UNSPECIFIED = 0,
  RAM_CPU = 1,
  RAM_GPU = 2,
  NVME = 3,
  SSD = 4,
  HDD = 5,
  CXL_MEMORY = 6,
  CXL_TYPE2_DEVICE = 7,
  CUSTOM = 999,
};
std::string_view to_string(StorageClass c) noexcept;
std::optional<StorageClass> parse_storage_class(std::string_view s) noexcept;
// Tier rank for demotion order: GPU(0) -> DRAM(1) -> CXL(2) -> NVMe(3) -> SSD(4) -> HDD(5).
int tier_rank(StorageClass c) noexcept;
bool is_disk_class(StorageClass c) noexcept;

// Data-plane endpoint of a worker (reference UcxEndpoint, types.h:97-102).  For host tiers this
// is the worker's TCP data server; for the GPU tier `worker_key` carries the fabric handle
// (CUDA IPC handle or VMM export descriptor) of the slab.
struct TransportEndpoint {
  std::string ip;
  uint32_t port = 0;
  std::vector<uint8_t> worker_key;
  bool operator==(const TransportEndpoint&) const = default;
};
using UcxEndpoint = TransportEndpoint;  // reference name

struct MemoryLocation {  // host memory reachable through the worker's data server
  uint64_t remote_addr = 0;
  uint32_t rkey = 0;
  uint64_t size = 0;
  bool operator==(const MemoryLocation&) const = default;
};
struct FileLocation {
  std::string file_path;
  uint64_t file_offset = 0;
  bool operator==(const FileLocation&) const = default;
};
struct CxlMemoryLocation {
  std::string device_id;
  uint64_t region_id = 0;
  uint64_t offset = 0;
  uint64_t size = 0;
  bool operator==(const CxlMemoryLocation&) const = default;
};
// An extent of a GPU worker's exported HBM slab: resolved by clients through the fabric's peer
// table to a peer-mapped (or NVLS multicast) virtual address.
struct GpuSlabLocation {
  uint32_t device_rank = 0;  // CUDA ordinal / worker rank inside the NVSwitch domain
  uint32_t slab_id = 0;
  uint64_t offset = 0;
  uint64_t size = 0;
  bool operator==(const GpuSlabLocation&) const = default;
};
using LocationDetail = std::variant<MemoryLocation, FileLocation, CxlMemoryLocation, GpuSlabLocation>;

struct ShardPlacement {
  MemoryPoolId pool_id;
  WorkerId worker_id;
  TransportEndpoint endpoint;
  StorageClass storage_class = StorageClass::STORAGE_UNSPECIFIED;
  uint64_t length = 0;
  LocationDetail location;
  uint64_t checksum = 0;  // digest of this shard's bytes, valid once the put completed
  ChecksumAlgo checksum_algo = ChecksumAlgo::NONE;
  bool operator==(const ShardPlacement&) const = default;
};

struct CopyPlacement {
  uint32_t copy_index = 0;
  std::vector<ShardPlacement> shards;
  size_t shards_size() const noexcept { return shards.size(); }
  bool operator==(const CopyPlacement&) const = default;
};

// Per-object placement / durability policy (reference WorkerConfig, types.h:161-187).
struct WorkerConfig {
  size_t replication_factor = DEFAULT_REPLICATION_FACTOR;
  size_t max_workers_per_copy = DEFAULT_MAX_WORKERS_PER_COPY;
  bool enable_soft_pin = false;
  std::string preferred_node;
  std::vector<StorageClass> preferred_classes;
  uint64_t ttl_ms = 30ull * 60 * 1000;  // 0 = never expires
  bool enable_locality_awareness = true;
  bool prefer_contiguous = false;
  size_t min_shard_size = 4096;
  // --- B200-native extensions
  ChecksumAlgo checksum = ChecksumAlgo::BBH64;
  bool pack_fp8 = false;          // store bf16 payload as block-scaled MXFP8 (E4M3 + E8M0/32)
  bool symmetric_replicas = false;  // same slab offset on every replica (NVLS multicast fan-out)
  bool operator==(const WorkerConfig&) const = default;
};
Json to_json(const WorkerConfig& c);
WorkerConfig worker_config_from_json(const Json& j);

struct ClusterStats {
  size_t total_workers = 0;
  size_t total_memory_pools = 0;
  size_t total_objects = 0;
  size_t total_capacity = 0;
  size_t used_capacity = 0;
  double avg_utilization = 0.0;
  // extensions
  size_t pending_objects = 0;
  size_t active_clients = 0;
  bool operator==(const ClusterStats&) const = default;
};
Json to_json(const ClusterStats& s);

struct KeystoneConfig {
  std::string cluster_id = DEFAULT_CLUSTER_ID;
  std::string etcd_endpoints;  // comma separated coordination endpoints ("" = in-process store)
  std::string listen_address = "0.0.0.0:9090";
  std::string http_metrics_port = "9091";
  std::string service_id;
  bool enable_gc = true;
  bool enable_ha = false;
  double eviction_ratio = 0.1;
  double high_watermark = DEFAULT_HIGH_WATERMARK;
  int64_t client_ttl_sec = DEFAULT_CLIENT_TTL_SEC;
  std::string auth_token;  // shared cluster token (net/tcp.h); empty = open cluster (BB_AUTH_TOKEN is the default)
  std::string auth_token_ro;       // second secret: members that prove only this one are read-only (net/tcp.h); BB_AUTH_TOKEN_RO
  bool encrypt_transport = false;  // AES-256-GCM on every RPC frame, keyed from the token (net/tcp.h secure mode); BB_ENCRYPT_TRANSPORT=1
  std::string http_auth_token;     // /metrics and /stats need `Authorization: Bearer <this>` (net/tcp.h); BB_HTTP_TOKEN
  std::string audit_log;           // append-only JSON-lines trail of security events and management calls (common/audit.h); BB_AUDIT_LOG
  std::string tenants_file;        // YAML table of tenants: own secret, key-prefix ACL, byte / object budget (common/tenant.h); BB_TENANTS_FILE
  int64_t worker_heartbeat_ttl_sec = 30;
  int64_t service_registration_ttl_sec = 60;
  int64_t service_refresh_interval_sec = 30;
  int64_t gc_interval_sec = 30;
  int64_t health_check_interval_sec = 10;
  int32_t max_replicas = 3;
  // > 0: the health loop compacts a pool (a few moves per round) whose fragmentation ratio exceeds this value
  double compaction_fragmentation_threshold = 0.0;
  // > 0: every health round re-hashes about this many objects at their workers and replaces copies that rotted (scrub);
  // the walk resumes where the last round stopped, so a full pass takes objects / scrub_objects_per_round rounds
  int32_t scrub_objects_per_round = 0;
  int32_t promote_after_reads = 0;    // > 0: an object read this often while it sits below the top tier is promoted back
  std::vector<TierRule> tier_policy;  // size-based class preference for puts that name no preferred class
  int32_t default_replicas = 1;
  // extensions
  int32_t rpc_threads = 2;
  int32_t rpc_busy_poll_us = 0;  // RPC threads poll without sleeping this long after a request (latency vs CPU)
  std::string log_level;  // from the `logging:` section the reference ignores
  std::string log_file;
  // Local metadata log (snapshot + append-only log, csrc/common/durable_log.h) of a single, non-HA Keystone: object
  // records are made durable under this directory before put_complete is acknowledged, and replayed on start.  HA
  // pairs log into the coordination store instead (fenced by the leader's term), so that the standby can resume.
  std::string wal_path;
  // Reservation protocol between Keystone and workers (keystone_service.h ReservationHooks): off by default -- the GPU
  // fast path is one-sided and a worker cannot police stores into its slab -- on for deployments that want worker-side
  // accounting of every shard and writer-crash cleanup by token expiry.
  bool enable_reservations = false;
  int64_t reservation_ttl_ms = 10 * 60 * 1000;  // reference: 10 minutes (ram_backend.cpp:69)
  bool wal_fsync = true;        // false: page-cache only (survives a process crash, not a power cut)
  int wal_snapshot_mb = 64;     // compact the log into a snapshot once it grows past this

  // Throws std::runtime_error on unreadable / invalid files (as the reference does).
  static KeystoneConfig from_yaml(const std::string& file_path);
  static Result<KeystoneConfig> from_json(const Json& root, std::string* err = nullptr);
  ErrorCode validate(std::string* err = nullptr) const;
};
Json to_json(const KeystoneConfig& c);

struct ClientConfig {
  std::string node_id;
  std::string keystone_address;
  std::string local_address = "0.0.0.0:0";
  size_t memory_pool_size = 1ull << 30;
  std::string storage_path;
};

// A worker's advertised memory pool (reference MemoryPool, types.h:464-493; JSON schema
// worker_service.cpp:494-516).  `ucx_*` names are kept in the JSON for schema parity.
struct MemoryPool {
  MemoryPoolId id;
  NodeId node_id;
  WorkerId worker_id;
  uint64_t base_addr = 0;
  uint64_t size = 0;
  uint64_t used = 0;
  StorageClass storage_class = StorageClass::STORAGE_UNSPECIFIED;
  std::string ucx_endpoint;      // "host:port" of the worker's data server
  uint64_t ucx_remote_addr = 0;  // base address clients add offsets to (host tiers)
  std::string ucx_rkey_hex;      // registration key: zero-padded hex, no separators
  // topology (consumed by the placement engine, unlike the reference: SURVEY §2.7)
  int32_t gpu_device_id = -1;
  int32_t numa_node = -1;
  double max_bw_gbps = 0.0;
  std::string fabric_domain;     // pools in the same NVSwitch domain can use fused P2P kernels
  std::string mount_path;        // disk tiers

  double utilization() const noexcept { return size ? static_cast<double>(used) / static_cast<double>(size) : 0.0; }
  uint64_t available() const noexcept { return size > used ? size - used : 0; }
  bool operator==(const MemoryPool&) const = default;
};
Json to_json(const MemoryPool& p);
Result<MemoryPool> memory_pool_from_json(const Json& j);

// Worker registration record (reference worker JSON, worker_service.cpp:479-492).
struct WorkerRecord {
  WorkerId worker_id;
  NodeId node_id;
  std::string rpc_endpoint;
  std::string ucx_endpoint;
  std::vector<std::string> interconnects;
  std::vector<StorageClass> storage_classes;
  double max_bw_gbps = 0.0;
  int32_t numa_node = -1;
  std::string version;
};
Json to_json(const WorkerRecord& w);
Result<WorkerRecord> worker_record_from_json(const Json& j);

// Hex helpers for registration keys: fixed 2 chars per byte (fixes reference bug §2.8 #7).
std::string bytes_to_hex(const std::vector<uint8_t>& b);
std::optional<std::vector<uint8_t>> hex_to_bytes(std::string_view hex);

// "host:port" -> (host, port); nullopt when malformed.
std::optional<std::pair<std::string, uint32_t>> split_host_port(std::string_view s);

UUID generate_uuid();
std::string uuid_to_string(const UUID& u);

}  // namespace bb

namespace std {
template <>
struct hash<bb::UUID> {
  size_t operator()(const bb::UUID& id) const noexcept {
    uint64_t a = id.first ^ (id.second + 0x9e3779b97f4a7c15ULL + (id.first << 6) + (id.first >> 2));
    a ^= a >> 33;
    a *= 0xff51afd7ed558ccdULL;
    a ^= a >> 33;
    return static_cast<size_t>(a);
  }
};
}  // namespace std
