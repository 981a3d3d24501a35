#include "common/trace.h"
#include "client/blackbird_client.h"

#include "common/tenant.h"
#include "common/mxfp8.h"
#include "common/tchash_def.h"

#include <algorithm>
#include <atomic>
#include <cstring>
#include <future>
#include <map>
#include <thread>

#include "common/log.h"
#include "rpc/wire.h"
#include "worker/worker_service.h"

namespace bb::client {

using keystone::PutStartItem;
using keystone::ShardChecksums;

namespace {
double us_since(TimePoint t0) { return std::chrono::duration<double, std::micro>(Clock::now() - t0).count(); }

// Runs fn(i) for i in [0, n) on up to `par` threads; returns the first error.
template <typename F>
ErrorCode parallel_for(size_t n, size_t par, F&& fn) {
  if (n == 0) return ErrorCode::OK;
  par = std::max<size_t>(1, std::min(par, n));
  if (par == 1) {
    for (size_t i = 0; i < n; ++i) {
      ErrorCode ec = fn(i);
      if (ec != ErrorCode::OK) return ec;
    }
    return ErrorCode::OK;
  }
  std::atomic<size_t> next{0};
  std::atomic<uint32_t> first_err{0};
  std::vector<std::thread> th;
  for (size_t t = 0; t < par; ++t)
    th.emplace_back([&] {
      while (first_err.load() == 0) {
        const size_t i = next.fetch_add(1);
        if (i >= n) break;
        ErrorCode ec = fn(i);
        if (ec != ErrorCode::OK) {
          uint32_t z = 0;
          first_err.compare_exchange_strong(z, static_cast<uint32_t>(ec));
        }
      }
    });
  for (auto& t : th) t.join();
  return static_cast<ErrorCode>(first_err.load());
}
}  // namespace

BlackbirdClient::BlackbirdClient(BlackbirdClientOptions opts) : opts_(std::move(opts)) {}
BlackbirdClient::BlackbirdClient(std::shared_ptr<rpc::KeystoneApi> keystone, BlackbirdClientOptions opts)
    : opts_(std::move(opts)), keystone_(std::move(keystone)) {
  if (keystone_) keystone_->set_identity(session_id_, opts_.node_id);
}
BlackbirdClient::~BlackbirdClient() {
  std::lock_guard<std::mutex> lk(shm_mu_);
  for (auto& [id, p] : shm_pools_) worker::unmap_shared_pool(p.base, p.size);
  shm_pools_.clear();
}

ErrorCode BlackbirdClient::connect() {
  if (!opts_.auth_token.empty()) net::set_cluster_token(opts_.auth_token);
  if (opts_.encrypt_transport) net::set_transport_encryption(true);
  if (!opts_.auth_token_ro.empty()) net::set_cluster_token_ro(opts_.auth_token_ro);
  if (!opts_.tenant.empty()) set_client_tenant(opts_.tenant, opts_.tenant_secret);
  if (!keystone_) {
    auto c = std::make_shared<rpc::KeystoneRpcClient>();
    c->set_timeout_ms(opts_.rpc_timeout_ms);
    const int connect_ms = std::min(opts_.rpc_timeout_ms, 5000);
    ErrorCode ec = opts_.keystone_endpoints.empty() ? c->connect(opts_.keystone_host, opts_.keystone_port, connect_ms)
                                                    : c->connect_any(opts_.keystone_endpoints, connect_ms);
    if (ec != ErrorCode::OK) return ec;
    keystone_ = c;
  }
  if (opts_.register_session) {
    auto s = keystone_->client_register(opts_.node_id);
    if (!s.ok()) return s.error();
    session_id_ = s.value();
  }
  keystone_->set_identity(session_id_, opts_.node_id);
  return ErrorCode::OK;
}

// ================================================================ worker connections
std::shared_ptr<net::RpcClient> BlackbirdClient::acquire(const std::string& endpoint) {
  {
    std::lock_guard<std::mutex> lk(conn_mu_);
    auto& v = idle_conns_[endpoint];
    if (!v.empty()) {
      auto c = v.back();
      v.pop_back();
      return c;
    }
  }
  auto hp = split_host_port(endpoint);
  if (!hp) return nullptr;
  auto c = std::make_shared<net::RpcClient>();
  if (c->connect(hp->first, static_cast<uint16_t>(hp->second), std::min(opts_.rpc_timeout_ms, 5000)) != ErrorCode::OK) return nullptr;
  c->set_bulk_buffers();
  return c;
}

void BlackbirdClient::release(const std::string& endpoint, std::shared_ptr<net::RpcClient> c) {
  if (!c || !c->connected()) return;
  std::lock_guard<std::mutex> lk(conn_mu_);
  auto& v = idle_conns_[endpoint];
  if (v.size() < 16) v.push_back(std::move(c));
}

uint64_t BlackbirdClient::shard_offset(const ShardPlacement& s) {
  if (auto* g = std::get_if<GpuSlabLocation>(&s.location)) return g->offset;
  if (auto* f = std::get_if<FileLocation>(&s.location)) return f->file_offset;
  if (auto* c = std::get_if<CxlMemoryLocation>(&s.location)) return c->offset;
  return 0;
}

namespace {
constexpr uint64_t kDataChunk = 8ull << 20;     // one D_WRITE / D_READ request
constexpr uint64_t kStreamMin = 4ull << 20;     // a shard is split over several connections from 2x this size

// Splits [0, len) into up to `par` ranges whose boundaries are multiples of the BBH64 tile (so per-range digests
// combine) and runs fn(range_begin, range_len, range_index) on one thread each.
template <typename F>
ErrorCode for_each_stream(uint64_t len, size_t par, F&& fn) {
  size_t n = static_cast<size_t>(std::min<uint64_t>(std::max<size_t>(par, 1), len / kStreamMin));
  if (n <= 1) return fn(0, len, 0);
  const uint64_t tiles = (len + tchash::kTileBytes - 1) / tchash::kTileBytes;
  const uint64_t per = (tiles + n - 1) / n * tchash::kTileBytes;
  n = static_cast<size_t>((len + per - 1) / per);
  std::vector<ErrorCode> ecs(n, ErrorCode::OK);
  std::vector<std::thread> th;
  for (size_t i = 1; i < n; ++i)
    th.emplace_back([&, i] { ecs[i] = fn(i * per, std::min<uint64_t>(per, len - i * per), i); });
  ecs[0] = fn(0, std::min<uint64_t>(per, len), 0);
  for (auto& t : th) t.join();
  for (ErrorCode ec : ecs)
    if (ec != ErrorCode::OK) return ec;
  return ErrorCode::OK;
}
// Hashes a byte range on its own thread while the transfer loop moves it: the loop publishes how far the bytes are
// valid (a put has them all from the start, a get as the chunks arrive) and collects the range digest at the end.
class RangeHasher {
 public:
  RangeHasher(ChecksumAlgo algo, const uint8_t* base, uint64_t shard_len, uint64_t begin, uint64_t len, bool all_valid)
      : algo_(algo), base_(base), shard_len_(shard_len), begin_(begin), len_(len), valid_(all_valid ? len : 0) {
    if (algo_ != ChecksumAlgo::NONE && len_ >= (1u << 20)) th_ = std::thread([this] { run(); });
    else inline_ = true;
  }
  ~RangeHasher() {
    abort_.store(true);
    if (th_.joinable()) th_.join();
  }
  void advance(uint64_t valid_len) { valid_.store(valid_len, std::memory_order_release); }
  // crc: CRC32C of the range (standard init / final xor, combinable with crc32c_combine); bbh: unfinalised tile sum
  void finish(uint32_t* crc, uint64_t* bbh) {
    valid_.store(len_, std::memory_order_release);
    if (inline_) run();
    else if (th_.joinable()) th_.join();
    *crc = crc_;
    *bbh = bbh_;
  }

 private:
  void run() {
    constexpr uint64_t kStep = 1ull << 20;  // multiple of the BBH64 tile
    uint64_t done = 0;
    while (done < len_) {
      uint64_t v = valid_.load(std::memory_order_acquire);
      if (v <= done) {
        if (abort_.load()) return;
        std::this_thread::yield();
        continue;
      }
      v = v == len_ ? len_ : v / kStep * kStep;  // whole steps (tile aligned) until the tail
      if (v <= done) {
        if (abort_.load()) return;
        std::this_thread::yield();
        continue;
      }
      const uint64_t n = std::min(kStep, v - done);
      if (algo_ == ChecksumAlgo::CRC32C) crc_ = crc32c(base_ + begin_ + done, n, crc_);
      else if (is_tile_sum(algo_))
        bbh_ += tile_sum_partial(algo_, base_, shard_len_, (begin_ + done) / tchash::kTileBytes, (n + tchash::kTileBytes - 1) / tchash::kTileBytes);
      done += n;
    }
  }
  ChecksumAlgo algo_;
  const uint8_t* base_;
  uint64_t shard_len_, begin_, len_;
  std::atomic<uint64_t> valid_;
  std::atomic<bool> abort_{false};
  bool inline_ = false;
  uint32_t crc_ = 0;
  uint64_t bbh_ = 0;
  std::thread th_;
};
}  // namespace

uint8_t* BlackbirdClient::shm_resolve(const ShardPlacement& s) {
  static const bool env_off = [] { const char* e = std::getenv("BB_DISABLE_SHM"); return e && *e && *e != '0'; }();
  if (!opts_.enable_shm || env_off || s.storage_class != StorageClass::RAM_CPU) return nullptr;
  const auto* loc = std::get_if<MemoryLocation>(&s.location);
  const auto& key = s.endpoint.worker_key;
  if (!loc || key.size() <= 5 || std::memcmp(key.data(), "file:", 5) != 0) return nullptr;
  {
    std::lock_guard<std::mutex> lk(shm_mu_);
    auto it = shm_pools_.find(s.pool_id);
    if (it != shm_pools_.end()) {
      if (it->second.key == key) {
        const ShmPool& p = it->second;
        if (loc->remote_addr < p.remote_base || loc->remote_addr - p.remote_base + s.length > p.size) return nullptr;
        return p.base + (loc->remote_addr - p.remote_base);
      }
      worker::unmap_shared_pool(it->second.base, it->second.size);  // the worker restarted: new memfd, new key
      shm_pools_.erase(it);
    }
    auto un = shm_unreachable_.find(s.pool_id);
    if (un != shm_unreachable_.end() && un->second == key) return nullptr;
  }
  // first shard in this pool: learn its geometry from the registry, then map it
  ShmPool p;
  auto pools = keystone_->get_memory_pools();
  if (pools.ok())
    for (const auto& mp : pools.value())
      if (mp.id == s.pool_id) {
        p.size = mp.size;
        p.remote_base = mp.ucx_remote_addr ? mp.ucx_remote_addr : mp.base_addr;
      }
  if (p.size) p.base = static_cast<uint8_t*>(worker::map_shared_pool(key, p.size));
  std::lock_guard<std::mutex> lk(shm_mu_);
  if (!p.base) {  // other host / pid namespace / user: stay on the data server
    shm_unreachable_[s.pool_id] = key;
    return nullptr;
  }
  p.key = key;
  auto [it, fresh] = shm_pools_.emplace(s.pool_id, p);
  if (!fresh) worker::unmap_shared_pool(p.base, p.size);  // another thread mapped it first
  else metrics_.inc("shm_pools_mapped_total");
  const ShmPool& q = it->second;
  if (loc->remote_addr < q.remote_base || loc->remote_addr - q.remote_base + s.length > q.size) return nullptr;
  return q.base + (loc->remote_addr - q.remote_base);
}

namespace {
// memcpy of a shard as up to `par` tile-aligned ranges on their own threads, each hashed while it is hot in cache.
struct ShmPart {
  uint32_t crc = 0;
  uint64_t len = 0;
  uint64_t bbh = 0;
};
uint64_t shm_copy(uint8_t* dst, const uint8_t* src, const uint8_t* hash_base, uint64_t len, size_t par, ChecksumAlgo algo) {
  if (algo == ChecksumAlgo::NONE) par = 1;  // a bare memcpy already runs at memory speed; threads only help the hashing
  std::vector<ShmPart> parts(std::max<size_t>(1, par));
  for_each_stream(len, par, [&](uint64_t begin, uint64_t n, size_t idx) -> ErrorCode {
    ShmPart& part = parts[idx];
    part.len = n;
    constexpr uint64_t kStep = 1ull << 20;  // copy + hash in cache-sized steps (multiple of the BBH64 tile)
    for (uint64_t o = begin; o < begin + n; o += kStep) {
      const uint64_t m = std::min(kStep, begin + n - o);
      std::memcpy(dst + o, src + o, m);
      if (algo == ChecksumAlgo::CRC32C) part.crc = crc32c(hash_base + o, m, part.crc);
      else if (is_tile_sum(algo))
        part.bbh += tile_sum_partial(algo, hash_base, len, o / tchash::kTileBytes, (m + tchash::kTileBytes - 1) / tchash::kTileBytes);
    }
    return ErrorCode::OK;
  });
  if (algo == ChecksumAlgo::CRC32C) {
    uint32_t crc = 0;
    bool first = true;
    for (const ShmPart& p : parts) {
      if (p.len == 0 && !first) continue;
      crc = first ? p.crc : crc32c_combine(crc, p.crc, p.len);
      first = false;
    }
    return crc;
  }
  if (is_tile_sum(algo)) {
    uint64_t sum = 0;
    for (const ShmPart& p : parts) sum += p.bbh;
    return tile_sum_finalize(sum, len);
  }
  return 0;
}
}  // namespace

ErrorCode BlackbirdClient::write_shard(const ShardPlacement& s, const uint8_t* src, uint64_t* digest, ChecksumAlgo algo) {
  if (uint8_t* mapped = shm_resolve(s)) {  // same host: one-sided write into the worker's pool
    const uint64_t d = shm_copy(mapped, src, src, s.length, opts_.io_parallelism, algo);
    if (digest) *digest = d;
    metrics_.inc("shm_put_shards_total");
    metrics_.inc("shm_put_bytes_total", s.length);
    return ErrorCode::OK;
  }
  const std::string ep = s.endpoint.ip + ":" + std::to_string(s.endpoint.port);
  uint64_t base_off = shard_offset(s);
  bool absolute = false;
  if (auto* m = std::get_if<MemoryLocation>(&s.location)) {
    base_off = m->remote_addr;  // absolute address; the worker subtracts its base
    absolute = true;
  }
  // Large shards go out as several streams (one connection + one thread each); every stream sends its range in
  // kDataChunk requests with a gathered write (header + bytes straight from the caller's buffer) and hashes it while the
  // worker stores the previous chunk.  Per-stream digests combine: CRC32C by shift algebra, BBH64 by addition.
  struct Part {
    uint32_t crc = 0;
    uint64_t len = 0;
    uint64_t bbh = 0;
  };
  std::vector<Part> parts(std::max<size_t>(1, opts_.io_parallelism));
  ErrorCode ec = for_each_stream(s.length, opts_.io_parallelism, [&](uint64_t begin, uint64_t len, size_t idx) -> ErrorCode {
    auto conn = acquire(ep);
    if (!conn) return ErrorCode::CONNECTION_FAILED;
    Part& part = parts[idx];
    part.len = len;
    RangeHasher hasher(algo, src, s.length, begin, len, /*all_valid=*/true);
    for (uint64_t pos = begin; pos < begin + len || (s.length == 0 && pos == 0); pos += kDataChunk) {
      const uint32_t n = static_cast<uint32_t>(std::min<uint64_t>(kDataChunk, begin + len - pos));
      wire::Writer w;
      w.str(s.pool_id);
      w.u64((base_off + pos) | (absolute ? (1ull << 63) : 0));
      w.u32(n);
      auto r = conn->call_gather(worker::D_WRITE, w.data(), src + pos, n, opts_.rpc_timeout_ms);
      if (!r.ok()) return ErrorCode::TRANSFER_FAILED;
      wire::Reader rd(r.value());
      const ErrorCode wec = rd.ec();
      if (wec != ErrorCode::OK) {
        release(ep, conn);
        return wec;
      }
      if (s.length == 0) break;
    }
    hasher.finish(&part.crc, &part.bbh);
    release(ep, conn);
    return ErrorCode::OK;
  });
  if (ec != ErrorCode::OK) return ec;
  if (digest) {
    if (algo == ChecksumAlgo::CRC32C) {
      uint32_t crc = 0;
      bool first = true;
      for (const Part& p : parts) {
        if (p.len == 0 && !first) continue;
        crc = first ? p.crc : crc32c_combine(crc, p.crc, p.len);
        first = false;
      }
      *digest = crc;
    } else if (is_tile_sum(algo)) {
      uint64_t sum = 0;
      for (const Part& p : parts) sum += p.bbh;
      *digest = tile_sum_finalize(sum, s.length);
    } else {
      *digest = 0;
    }
  }
  return ErrorCode::OK;
}

ErrorCode BlackbirdClient::read_shard(const ShardPlacement& s, uint8_t* dst, ChecksumAlgo algo) {
  if (const uint8_t* mapped = shm_resolve(s)) {  // same host: one-sided read out of the worker's pool
    const bool check = algo != ChecksumAlgo::NONE && s.checksum_algo == algo;
    const uint64_t got = shm_copy(dst, mapped, dst, s.length, opts_.io_parallelism, check ? algo : ChecksumAlgo::NONE);
    metrics_.inc("shm_get_shards_total");
    metrics_.inc("shm_get_bytes_total", s.length);
    if (check && got != s.checksum) {
      metrics_.inc("checksum_mismatch_total");
      return ErrorCode::CHECKSUM_MISMATCH;
    }
    return ErrorCode::OK;
  }
  const std::string ep = s.endpoint.ip + ":" + std::to_string(s.endpoint.port);
  uint64_t base_off = shard_offset(s);
  bool absolute = false;
  if (auto* m = std::get_if<MemoryLocation>(&s.location)) {
    base_off = m->remote_addr;
    absolute = true;
  }
  const bool verify = algo != ChecksumAlgo::NONE && s.checksum_algo == algo;
  struct Part {
    uint32_t crc = 0;
    uint64_t len = 0;
    uint64_t bbh = 0;
  };
  std::vector<Part> parts(std::max<size_t>(1, opts_.io_parallelism));
  // Same streams as write_shard; the response payload is received straight into the caller's buffer.
  ErrorCode ec = for_each_stream(s.length, opts_.io_parallelism, [&](uint64_t begin, uint64_t len, size_t idx) -> ErrorCode {
    auto conn = acquire(ep);
    if (!conn) return ErrorCode::CONNECTION_FAILED;
    Part& part = parts[idx];
    part.len = len;
    RangeHasher hasher(verify ? algo : ChecksumAlgo::NONE, dst, s.length, begin, len, /*all_valid=*/false);
    for (uint64_t pos = begin; pos < begin + len; pos += kDataChunk) {
      const uint32_t n = static_cast<uint32_t>(std::min<uint64_t>(kDataChunk, begin + len - pos));
      wire::Writer w;
      w.str(s.pool_id);
      w.u64((base_off + pos) | (absolute ? (1ull << 63) : 0));
      w.u32(n);
      size_t got = 0;
      auto r = conn->call_scatter(worker::D_READ, w.data(), 4, dst + pos, n, &got, opts_.rpc_timeout_ms);
      if (!r.ok()) return ErrorCode::TRANSFER_FAILED;
      if (r.value().size() < 4) return ErrorCode::TRANSFER_FAILED;
      uint32_t e;
      std::memcpy(&e, r.value().data(), 4);
      if (e != 0) {
        release(ep, conn);
        return static_cast<ErrorCode>(e);
      }
      if (got != n) return ErrorCode::TRANSFER_FAILED;
      hasher.advance(pos + n - begin);
    }
    hasher.finish(&part.crc, &part.bbh);
    release(ep, conn);
    return ErrorCode::OK;
  });
  if (ec != ErrorCode::OK) return ec;
  if (verify) {
    uint64_t got = 0;
    if (algo == ChecksumAlgo::CRC32C) {
      uint32_t crc = 0;
      bool first = true;
      for (const Part& p : parts) {
        if (p.len == 0 && !first) continue;
        crc = first ? p.crc : crc32c_combine(crc, p.crc, p.len);
        first = false;
      }
      got = crc;
    } else {
      uint64_t sum = 0;
      for (const Part& p : parts) sum += p.bbh;
      got = bbh64_finalize(sum, s.length);
    }
    if (got != s.checksum) {
      metrics_.inc("checksum_mismatch_total");
      return ErrorCode::CHECKSUM_MISMATCH;
    }
  }
  return ErrorCode::OK;
}

ErrorCode BlackbirdClient::transfer_put(const std::vector<CopyPlacement>& copies, const uint8_t* data, ChecksumAlgo algo,
                                        ShardChecksums* sums) {
  struct Job {
    size_t c, s;
    uint64_t off;
  };
  std::vector<Job> jobs;
  sums->assign(copies.size(), {});
  for (size_t c = 0; c < copies.size(); ++c) {
    uint64_t off = 0;
    (*sums)[c].assign(copies[c].shards.size(), 0);
    for (size_t s = 0; s < copies[c].shards.size(); ++s) {
      jobs.push_back({c, s, off});
      off += copies[c].shards[s].length;  // the source offset is the running shard offset (bug #8)
    }
  }
  return parallel_for(jobs.size(), opts_.io_parallelism, [&](size_t i) {
    const Job& j = jobs[i];
    return write_shard(copies[j.c].shards[j.s], data + j.off, &(*sums)[j.c][j.s], algo);
  });
}

ErrorCode BlackbirdClient::transfer_get(const std::vector<CopyPlacement>& copies, uint8_t* dst, size_t size) {
  ErrorCode last = ErrorCode::NO_COMPLETE_WORKER;
  for (const auto& copy : copies) {  // replica fail-over (reference reads copy 0 only, :283-287)
    uint64_t total = 0;
    for (const auto& s : copy.shards) total += s.length;
    if (total != size) {
      last = ErrorCode::DATA_CORRUPTION;
      continue;
    }
    std::vector<uint64_t> offs(copy.shards.size());
    uint64_t off = 0;
    for (size_t s = 0; s < copy.shards.size(); ++s) {
      offs[s] = off;
      off += copy.shards[s].length;
    }
    last = parallel_for(copy.shards.size(), opts_.io_parallelism, [&](size_t s) {
      return read_shard(copy.shards[s], dst + offs[s], copy.shards[s].checksum_algo);
    });
    if (last == ErrorCode::OK) return ErrorCode::OK;
    metrics_.inc("replica_failover_total");
    BB_LOG(WARNING) << "get: copy " << copy.copy_index << " failed with " << to_string(last) << ", trying next replica";
  }
  return last;
}

// ================================================================ reference API
Result<bool> BlackbirdClient::object_exists(const ObjectKey& key) {
  if (!keystone_) return ErrorCode::CLIENT_DISCONNECTED;
  return keystone_->object_exists(key);
}

Result<std::vector<CopyPlacement>> BlackbirdClient::get_workers(const ObjectKey& key) {
  if (!keystone_) return ErrorCode::CLIENT_DISCONNECTED;
  return keystone_->get_workers(key);
}

ErrorCode BlackbirdClient::put(const ObjectKey& key, const uint8_t* data, size_t size, const WorkerConfig& cfg) {
  if (!keystone_) return ErrorCode::CLIENT_DISCONNECTED;
  if (!data && size) return ErrorCode::INVALID_PARAMETERS;
  auto* ha = dynamic_cast<rpc::KeystoneRpcClient*>(keystone_.get());
  const uint64_t failovers = ha ? ha->failovers() : 0;
  ErrorCode ec = put_once(key, data, size, cfg);
  // The keystone failed over in the middle of this put: only completed objects are in the metadata log, so the new
  // leader has never heard of our pending one and put_complete comes back OBJECT_NOT_FOUND.  The bytes are still in
  // hand -- start over against the new leader instead of handing the caller an error that is not theirs.
  if (ec == ErrorCode::OBJECT_NOT_FOUND && ha && ha->failovers() != failovers) {
    metrics_.inc("put_restarted_after_failover_total");
    ec = put_once(key, data, size, cfg);
  }
  return ec;
}

ErrorCode BlackbirdClient::put_once(const ObjectKey& key, const uint8_t* data, size_t size, const WorkerConfig& cfg) {
  const TimePoint t0 = Clock::now();
  BB_TRACE_SPAN("client.put", size);
  auto placed = keystone_->put_start(key, size, cfg);
  if (!placed.ok()) return placed.error();
  ShardChecksums sums;
  ErrorCode ec = transfer_put(placed.value(), data, cfg.checksum, &sums);
  if (ec != ErrorCode::OK) {
    keystone_->put_cancel(key);
    metrics_.inc("put_failed_total");
    return ec;
  }
  ec = keystone_->put_complete(key, sums);
  if (ec == ErrorCode::OK) {
    metrics_.inc("put_total");
    metrics_.inc("put_bytes_total", size);
    metrics_.observe("put_latency_us", us_since(t0));
  }
  return ec;
}

// A transfer can lose a race with the Keystone moving the object (tier demotion / promotion, migrate_object, pool
// compaction, repair): the placements it holds were swapped and their extents re-used, which shows up as a digest
// mismatch or a failed read.  Fresh placements that differ from the ones just tried are worth one more attempt.
ErrorCode BlackbirdClient::get_with_refresh(const ObjectKey& key, uint8_t* (*alloc)(void*, size_t), void* ctx, size_t capacity, size_t* out_size) {
  Result<std::vector<CopyPlacement>> copies = keystone_->get_workers(key);
  ErrorCode ec = ErrorCode::OK;
  bool reread_same = false;
  for (int attempt = 0; attempt < 3; ++attempt) {
    if (!copies.ok()) return copies.error();
    if (copies.value().empty()) return ErrorCode::NO_COMPLETE_WORKER;
    size_t size = 0;
    for (const auto& s : copies.value().front().shards) size += s.length;
    if (out_size) *out_size = size;
    if (size > capacity) return ErrorCode::BUFFER_OVERFLOW;
    uint8_t* dst = alloc(ctx, size);
    ec = transfer_get(copies.value(), dst, size);
    if (ec == ErrorCode::OK) return ec;
    auto again = keystone_->get_workers(key);
    if (!again.ok()) return again.error();              // removed (or being re-written) meanwhile: that is the answer
    if (again.value() == copies.value()) {
      // Same placements.  A digest mismatch can still be a race -- the key was removed and re-put onto the very same
      // extent (first fit) and we read it half-written -- so that gets one more read; anything else is real.
      if (ec != ErrorCode::CHECKSUM_MISMATCH || reread_same) return ec;
      reread_same = true;
    }
    metrics_.inc("get_placement_refresh_total");
    copies = std::move(again);
  }
  return ec;
}

Result<std::vector<uint8_t>> BlackbirdClient::get(const ObjectKey& key) {
  if (!keystone_) return ErrorCode::CLIENT_DISCONNECTED;
  const TimePoint t0 = Clock::now();
  BB_TRACE_SPAN("client.get");
  std::vector<uint8_t> buf;
  size_t size = 0;
  ErrorCode ec = get_with_refresh(key, [](void* c, size_t n) {
    auto* v = static_cast<std::vector<uint8_t>*>(c);
    v->resize(n);
    return v->data();
  }, &buf, ~size_t{0}, &size);
  if (ec != ErrorCode::OK) return ec;
  metrics_.inc("get_total");
  metrics_.inc("get_bytes_total", size);
  metrics_.observe("get_latency_us", us_since(t0));
  return buf;
}

ErrorCode BlackbirdClient::get_into(const ObjectKey& key, void* buf, size_t capacity, size_t* out_size) {
  if (!keystone_) return ErrorCode::CLIENT_DISCONNECTED;
  return get_with_refresh(key, [](void* c, size_t) { return static_cast<uint8_t*>(c); }, buf, capacity, out_size);
}

ErrorCode BlackbirdClient::remove(const ObjectKey& key) {
  if (!keystone_) return ErrorCode::CLIENT_DISCONNECTED;
  return keystone_->remove_object(key);
}

// ================================================================ fused MXFP8 device API
std::vector<ErrorCode> BlackbirdClient::batch_put_device_fp8(const std::vector<ObjectKey>& keys, const std::vector<const void*>& bf16_ptrs,
                                                             const std::vector<uint64_t>& n_elems, const WorkerConfig& cfg, void* stream) {
  std::vector<ErrorCode> out(keys.size(), ErrorCode::INVALID_PARAMETERS);
  if (!keystone_) return std::vector<ErrorCode>(keys.size(), ErrorCode::CLIENT_DISCONNECTED);
  if (!device_) return std::vector<ErrorCode>(keys.size(), ErrorCode::NOT_IMPLEMENTED);
  if (bf16_ptrs.size() != keys.size() || n_elems.size() != keys.size()) return out;
  BB_TRACE_SPAN("batch_put_device_fp8", keys.size());
  WorkerConfig c = cfg;
  c.replication_factor = std::max<size_t>(1, std::min<size_t>(cfg.replication_factor, 3));  // one tile pass fans out to <= 3 copies
  c.max_workers_per_copy = 1;    // payload + scales of an object stay in one shard
  c.checksum = ChecksumAlgo::BBH64;
  c.pack_fp8 = true;
  if (c.preferred_classes.empty()) c.preferred_classes = {StorageClass::RAM_GPU};
  std::vector<PutStartItem> items;
  for (size_t i = 0; i < keys.size(); ++i) {
    if (!device_->fp8_eligible(n_elems[i])) return out;
    items.push_back(PutStartItem{keys[i], static_cast<size_t>(n_elems[i] + n_elems[i] / 32), c});
  }
  auto placed = keystone_->batch_put_start(items);
  std::vector<DeviceFp8Op> ops;
  std::vector<size_t> idx;
  for (size_t i = 0; i < keys.size(); ++i) {
    if (!placed[i].ok()) {
      out[i] = placed[i].error();
      continue;
    }
    const auto& copies = placed[i].value();
    bool fits = !copies.empty() && copies.size() <= 3;
    for (const auto& cp : copies) fits = fits && cp.shards.size() == 1 && device_->can_reach(cp.shards[0]);
    if (!fits) {
      keystone_->put_cancel(keys[i]);
      out[i] = ErrorCode::NOT_IMPLEMENTED;  // a copy is not a single GPU-fabric shard: caller packs + puts instead
      continue;
    }
    DeviceFp8Op op{&copies[0].shards[0], const_cast<void*>(bf16_ptrs[i]), n_elems[i], {}};
    for (size_t cidx = 1; cidx < copies.size(); ++cidx) op.replicas.push_back(&copies[cidx].shards[0]);
    ops.push_back(std::move(op));
    idx.push_back(i);
  }
  std::vector<uint64_t> digests;
  ErrorCode ec = ops.empty() ? ErrorCode::OK : device_->put_fp8(ops, stream, &digests);
  std::vector<ObjectKey> done;
  std::vector<ShardChecksums> sums;
  for (size_t k = 0; k < idx.size(); ++k) {
    if (ec != ErrorCode::OK || digests.size() != idx.size()) {
      keystone_->put_cancel(keys[idx[k]]);
      out[idx[k]] = ec != ErrorCode::OK ? ec : ErrorCode::INTERNAL_ERROR;
      continue;
    }
    done.push_back(keys[idx[k]]);
    sums.push_back(ShardChecksums(placed[idx[k]].value().size(), std::vector<uint64_t>{digests[k]}));  // same bytes in every copy
  }
  if (!done.empty()) {
    auto r = keystone_->batch_put_complete(done, sums);
    size_t j = 0;
    for (size_t k = 0; k < idx.size(); ++k)
      if (out[idx[k]] == ErrorCode::INVALID_PARAMETERS) out[idx[k]] = r[j++];
  }
  metrics_.inc("device_put_fp8_batches_total");
  return out;
}

std::vector<ErrorCode> BlackbirdClient::batch_get_device_fp8(const std::vector<ObjectKey>& keys, const std::vector<void*>& bf16_ptrs,
                                                             const std::vector<uint64_t>& n_elems, void* stream) {
  std::vector<ErrorCode> out(keys.size(), ErrorCode::INVALID_PARAMETERS);
  if (!keystone_) return std::vector<ErrorCode>(keys.size(), ErrorCode::CLIENT_DISCONNECTED);
  if (!device_) return std::vector<ErrorCode>(keys.size(), ErrorCode::NOT_IMPLEMENTED);
  if (bf16_ptrs.size() != keys.size() || n_elems.size() != keys.size()) return out;
  BB_TRACE_SPAN("batch_get_device_fp8", keys.size());
  auto placed = keystone_->batch_get_workers(keys);
  std::vector<std::vector<size_t>> candidates(keys.size());
  std::vector<size_t> idx;
  for (size_t i = 0; i < keys.size(); ++i) {
    if (!placed[i].ok()) {
      out[i] = placed[i].error();
      continue;
    }
    const auto& copies = placed[i].value();
    const uint64_t packed = n_elems[i] + n_elems[i] / 32;
    // usable copies: single GPU-fabric shard holding the whole packed object with a BBH64 digest; a copy in this
    // client's own HBM first, the others in hashed order (readers spread over the replicas)
    std::vector<size_t> order;
    const size_t start = copies.empty() ? 0 : std::hash<std::string>{}(opts_.node_id + keys[i]) % copies.size();
    for (int pass = 0; pass < 2; ++pass)
      for (size_t k = 0; k < copies.size(); ++k) {
        const size_t cidx = (start + k) % copies.size();
        const auto& cp = copies[cidx];
        if (cp.shards.size() != 1 || cp.shards[0].length != packed || cp.shards[0].checksum_algo != ChecksumAlgo::BBH64) continue;
        if (!device_->can_reach(cp.shards[0]) || device_->is_local(cp.shards[0]) != (pass == 0)) continue;
        order.push_back(cidx);
      }
    if (!device_->fp8_eligible(n_elems[i]) || order.empty()) {
      out[i] = ErrorCode::NOT_IMPLEMENTED;  // demoted to a host tier, striped, other digest: caller gets + unpacks instead
      continue;
    }
    candidates[i] = std::move(order);
    idx.push_back(i);
  }
  // one fused launch per attempt; objects whose digest did not verify are retried on their next replica
  std::vector<size_t> todo = idx;
  for (size_t attempt = 0; !todo.empty(); ++attempt) {
    std::vector<DeviceFp8Op> ops;
    std::vector<size_t> cur;
    for (size_t i : todo) {
      if (attempt >= candidates[i].size()) {
        out[i] = ErrorCode::CHECKSUM_MISMATCH;
        continue;
      }
      ops.push_back(DeviceFp8Op{&placed[i].value()[candidates[i][attempt]].shards[0], bf16_ptrs[i], n_elems[i], {}});
      cur.push_back(i);
    }
    if (ops.empty()) break;
    if (attempt > 0) metrics_.inc("replica_failover_total");
    std::vector<uint32_t> status;
    ErrorCode ec = device_->get_fp8(ops, stream, &status);
    todo.clear();
    for (size_t k = 0; k < cur.size(); ++k) {
      if (ec != ErrorCode::OK || status.size() != cur.size()) out[cur[k]] = ec != ErrorCode::OK ? ec : ErrorCode::INTERNAL_ERROR;
      else if (status[k]) todo.push_back(cur[k]);
      else out[cur[k]] = ErrorCode::OK;
    }
  }
  // Same rule as batch_get_device: a digest mismatch on every replica can mean the object was moved under us (tier
  // move, compaction, repair).  Keys whose placements changed since we read them get one more pass; a key that moved
  // to a non-fusable placement comes back NOT_IMPLEMENTED from that pass, i.e. "get + unpack instead".
  static thread_local int fp8_refresh_depth = 0;
  if (fp8_refresh_depth < 2) {
    std::vector<size_t> bad;
    for (size_t i = 0; i < keys.size(); ++i)
      if (out[i] == ErrorCode::CHECKSUM_MISMATCH && placed[i].ok()) bad.push_back(i);
    if (!bad.empty()) {
      std::vector<ObjectKey> bkeys;
      for (size_t i : bad) bkeys.push_back(keys[i]);
      auto again = keystone_->batch_get_workers(bkeys);
      std::vector<ObjectKey> rkeys;
      std::vector<void*> rptrs;
      std::vector<uint64_t> rn;
      std::vector<size_t> ridx;
      for (size_t k = 0; k < bad.size(); ++k) {
        const size_t i = bad[k];
        if (!again[k].ok()) out[i] = again[k].error();
        // changed placements, or (once) the same ones: a remove + re-put can land on the very same extent and be read half-written
        else if (!(again[k].value() == placed[i].value()) || fp8_refresh_depth == 0) rkeys.push_back(keys[i]), rptrs.push_back(bf16_ptrs[i]), rn.push_back(n_elems[i]), ridx.push_back(i);
      }
      if (!rkeys.empty()) {
        metrics_.inc("get_placement_refresh_total", rkeys.size());
        ++fp8_refresh_depth;
        auto recs = batch_get_device_fp8(rkeys, rptrs, rn, stream);
        --fp8_refresh_depth;
        for (size_t k = 0; k < ridx.size(); ++k) out[ridx[k]] = recs[k];
      }
    }
  }
  metrics_.inc("device_get_fp8_batches_total");
  return out;
}

ErrorCode BlackbirdClient::migrate(const ObjectKey& key, StorageClass target) {
  if (!keystone_) return ErrorCode::CLIENT_DISCONNECTED;
  return keystone_->migrate_object(key, target);
}

Result<ClusterStats> BlackbirdClient::cluster_stats() {
  if (!keystone_) return ErrorCode::CLIENT_DISCONNECTED;
  return keystone_->get_cluster_stats();
}

// ================================================================ batched host API
std::vector<ErrorCode> BlackbirdClient::batch_put(const std::vector<ObjectKey>& keys, const std::vector<const uint8_t*>& data,
                                                  const std::vector<size_t>& sizes, const WorkerConfig& cfg) {
  std::vector<ErrorCode> out(keys.size(), ErrorCode::INVALID_PARAMETERS);
  if (!keystone_) return std::vector<ErrorCode>(keys.size(), ErrorCode::CLIENT_DISCONNECTED);
  if (data.size() != keys.size() || sizes.size() != keys.size()) return out;
  std::vector<PutStartItem> items(keys.size());
  for (size_t i = 0; i < keys.size(); ++i) items[i] = PutStartItem{keys[i], sizes[i], cfg};
  auto placed = keystone_->batch_put_start(items);  // ONE control-plane round trip for the batch
  std::vector<ShardChecksums> sums(keys.size());
  std::vector<ObjectKey> done_keys, cancel_keys;
  std::vector<ShardChecksums> done_sums;
  std::vector<size_t> done_idx;
  parallel_for(keys.size(), opts_.io_parallelism, [&](size_t i) {
    if (!placed[i].ok()) {
      out[i] = placed[i].error();
      return ErrorCode::OK;
    }
    out[i] = transfer_put(placed[i].value(), data[i], cfg.checksum, &sums[i]);
    return ErrorCode::OK;
  });
  for (size_t i = 0; i < keys.size(); ++i) {
    if (!placed[i].ok()) continue;
    if (out[i] == ErrorCode::OK) {
      done_keys.push_back(keys[i]);
      done_sums.push_back(std::move(sums[i]));
      done_idx.push_back(i);
    } else {
      cancel_keys.push_back(keys[i]);
    }
  }
  if (!cancel_keys.empty()) keystone_->batch_put_cancel(cancel_keys);
  if (!done_keys.empty()) {
    auto ecs = keystone_->batch_put_complete(done_keys, done_sums);
    for (size_t k = 0; k < done_idx.size(); ++k) out[done_idx[k]] = ecs[k];
  }
  return out;
}

std::vector<Result<std::vector<uint8_t>>> BlackbirdClient::batch_get(const std::vector<ObjectKey>& keys) {
  std::vector<Result<std::vector<uint8_t>>> out(keys.size(), Result<std::vector<uint8_t>>(ErrorCode::CLIENT_DISCONNECTED));
  if (!keystone_) return out;
  auto placed = keystone_->batch_get_workers(keys);
  parallel_for(keys.size(), opts_.io_parallelism, [&](size_t i) {
    if (!placed[i].ok()) {
      out[i] = placed[i].error();
      return ErrorCode::OK;
    }
    if (placed[i].value().empty()) {
      out[i] = ErrorCode::NO_COMPLETE_WORKER;
      return ErrorCode::OK;
    }
    size_t size = 0;
    for (const auto& s : placed[i].value().front().shards) size += s.length;
    std::vector<uint8_t> buf(size);
    ErrorCode ec = transfer_get(placed[i].value(), buf.data(), size);
    if (ec == ErrorCode::OK) out[i] = std::move(buf);
    else out[i] = ec;
    return ErrorCode::OK;
  });
  return out;
}

std::vector<ErrorCode> BlackbirdClient::batch_remove(const std::vector<ObjectKey>& keys) {
  if (!keystone_) return std::vector<ErrorCode>(keys.size(), ErrorCode::CLIENT_DISCONNECTED);
  const TimePoint t0 = Clock::now();
  auto r = keystone_->batch_remove_object(keys);
  metrics_.observe("phase_remove_us", us_since(t0));
  return r;
}

std::vector<Result<bool>> BlackbirdClient::batch_exists(const std::vector<ObjectKey>& keys) {
  if (!keystone_) return std::vector<Result<bool>>(keys.size(), Result<bool>(ErrorCode::CLIENT_DISCONNECTED));
  return keystone_->batch_object_exists(keys);
}

// ================================================================ batched device API
std::vector<std::pair<size_t, size_t>> BlackbirdClient::plan_chunks(const std::vector<size_t>& sizes, double rpc_us_per_object) const {
  std::vector<std::pair<size_t, size_t>> chunks;
  uint64_t total = 0;
  for (size_t s : sizes) total += s;
  constexpr uint64_t kMinChunk = 256ull << 20;  // below this a chunk's kernel is too short to hide an RPC
  constexpr double kLaunchPenaltyUs = 120.0;    // measured: ramp + tail + launch gap + result read-back of one more fused launch
  const size_t depth = device_ ? device_->max_in_flight() : 1;
  size_t want = 1;
  if (depth >= 2 && sizes.size() >= 2 && total >= 2 * kMinChunk) {
    if (pipeline_chunks_ > 0) {
      want = pipeline_chunks_;
    } else {
      // Splitting hides (1 - 1/c) of the control-plane time behind kernels and costs (c - 1) launch penalties.
      // An in-process Keystone (tens of us per batch) is not worth a split; a remote one (100s of us) is.
      const double rpc_us = rpc_us_per_object * static_cast<double>(sizes.size());
      double best = 0;
      for (size_t c : {size_t{2}, size_t{4}}) {
        const double gain = rpc_us * (1.0 - 1.0 / static_cast<double>(c)) - static_cast<double>(c - 1) * kLaunchPenaltyUs;
        if (gain > best) best = gain, want = c;
      }
    }
    want = std::min<size_t>({want, static_cast<size_t>(total / kMinChunk), sizes.size()});
  }
  if (want <= 1) {
    chunks.emplace_back(0, sizes.size());
    return chunks;
  }
  const uint64_t target = total / want;
  size_t begin = 0;
  uint64_t acc = 0;
  for (size_t i = 0; i < sizes.size(); ++i) {
    acc += sizes[i];
    if (acc >= target && i + 1 < sizes.size() && chunks.size() + 1 < want) {
      chunks.emplace_back(begin, i + 1);
      begin = i + 1;
      acc = 0;
    }
  }
  chunks.emplace_back(begin, sizes.size());
  return chunks;
}

static void ewma_update(std::atomic<double>& v, double sample) {
  const double old = v.load(std::memory_order_relaxed);
  v.store(old == 0 ? sample : 0.75 * old + 0.25 * sample, std::memory_order_relaxed);
}

// Segment table entries one chunk of a segmented batch may hand to the transport (one fused launch each).
static constexpr size_t kMaxChunkSegments = size_t{1} << 20;

// Splits chunks further so that none carries more than kMaxChunkSegments segments (a chunk keeps at least one object).
static std::vector<std::pair<size_t, size_t>> cap_chunk_segments(const std::vector<std::pair<size_t, size_t>>& plan,
                                                                 const std::vector<size_t>& count) {
  std::vector<std::pair<size_t, size_t>> out;
  for (const auto& [b, e] : plan) {
    size_t begin = b, acc = 0;
    for (size_t i = b; i < e; ++i) {
      if (i > begin && acc + count[i] > kMaxChunkSegments) {
        out.emplace_back(begin, i);
        begin = i, acc = 0;
      }
      acc += count[i];
    }
    out.emplace_back(begin, e);
  }
  return out;
}

// Checks the segment rules object by object.  verdict[i] = OK for a valid object (its total length in total[i]); false
// when seg_counts do not add up to segs.size() (the whole batch is invalid).
static bool index_segments(const std::vector<DeviceSegment>& segs, const std::vector<uint32_t>& seg_counts, std::vector<size_t>* first,
                           std::vector<ErrorCode>* verdict, std::vector<size_t>* total) {
  uint64_t sum = 0;
  for (uint32_t c : seg_counts) sum += c;
  if (sum != segs.size()) return false;
  first->assign(seg_counts.size(), 0);
  total->assign(seg_counts.size(), 0);
  size_t pos = 0;
  for (size_t i = 0; i < seg_counts.size(); ++i) {
    const size_t n = seg_counts[i];
    (*first)[i] = pos;
    bool ok = n > 0;
    uint64_t bytes = 0;
    for (size_t k = 0; k < n && ok; ++k) {
      const DeviceSegment& s = segs[pos + k];
      ok = (s.ptr & 15) == 0 && s.len > 0 && (k + 1 == n || (s.len & 15) == 0);
      bytes += s.len;
    }
    pos += n;
    (*verdict)[i] = !ok ? ErrorCode::INVALID_PARAMETERS
                    : n > BlackbirdClient::kMaxObjectSegments ? ErrorCode::VALUE_OUT_OF_RANGE : ErrorCode::OK;
    (*total)[i] = bytes;
  }
  return true;
}

std::vector<ErrorCode> BlackbirdClient::batch_put_device(const std::vector<ObjectKey>& keys, const std::vector<const void*>& dev_ptrs,
                                                         const std::vector<size_t>& sizes, const WorkerConfig& cfg, void* stream) {
  return put_device_impl(keys, dev_ptrs, sizes, nullptr, cfg, stream);
}

std::vector<ErrorCode> BlackbirdClient::batch_put_device_gather(const std::vector<ObjectKey>& keys, const std::vector<DeviceSegment>& segs,
                                                                const std::vector<uint32_t>& seg_counts, const WorkerConfig& cfg,
                                                                void* stream) {
  std::vector<ErrorCode> out(keys.size(), ErrorCode::INVALID_PARAMETERS);
  if (!keystone_) return std::vector<ErrorCode>(keys.size(), ErrorCode::CLIENT_DISCONNECTED);
  if (!device_) return std::vector<ErrorCode>(keys.size(), ErrorCode::NOT_IMPLEMENTED);
  std::vector<size_t> first, total;
  if (seg_counts.size() != keys.size() || !index_segments(segs, seg_counts, &first, &out, &total))
    return std::vector<ErrorCode>(keys.size(), ErrorCode::INVALID_PARAMETERS);
  // the valid objects go on as one batch; the others keep their verdict
  SegView sv;
  sv.segs = segs.data();
  std::vector<ObjectKey> vkeys;
  std::vector<size_t> idx, sizes;
  for (size_t i = 0; i < keys.size(); ++i) {
    if (out[i] != ErrorCode::OK) continue;
    idx.push_back(i), vkeys.push_back(keys[i]), sizes.push_back(total[i]);
    sv.first.push_back(first[i]), sv.count.push_back(seg_counts[i]);
  }
  if (idx.empty()) return out;
  auto r = put_device_impl(vkeys, std::vector<const void*>(idx.size(), nullptr), sizes, &sv, cfg, stream);
  for (size_t k = 0; k < idx.size(); ++k) out[idx[k]] = r[k];
  return out;
}

std::vector<ErrorCode> BlackbirdClient::put_device_impl(const std::vector<ObjectKey>& keys, const std::vector<const void*>& dev_ptrs,
                                                        const std::vector<size_t>& sizes, const SegView* sv, const WorkerConfig& cfg,
                                                        void* stream) {
  std::vector<ErrorCode> out(keys.size(), ErrorCode::INVALID_PARAMETERS);
  if (!keystone_) return std::vector<ErrorCode>(keys.size(), ErrorCode::CLIENT_DISCONNECTED);
  if (!device_) return std::vector<ErrorCode>(keys.size(), ErrorCode::NOT_IMPLEMENTED);
  if (dev_ptrs.size() != keys.size() || sizes.size() != keys.size()) return out;
  const TimePoint t_all = Clock::now();
  BB_TRACE_SPAN("batch_put_device", keys.size());

  struct Chunk {
    size_t begin = 0, end = 0;
    std::vector<Result<std::vector<CopyPlacement>>> placed;
    std::vector<DeviceShardOp> ops;
    uint64_t ticket = 0;
    bool submitted = false;
    ErrorCode submit_error = ErrorCode::OK;
  };
  auto plan = plan_chunks(sizes, put_rpc_us_per_obj_.load(std::memory_order_relaxed));
  if (sv) plan = cap_chunk_segments(plan, sv->count);
  double rpc_us_total = 0;
  std::vector<Chunk> chunks(plan.size());
  std::vector<size_t> host_put;                      // objects whose placement is not on the GPU fabric
  std::map<size_t, std::vector<CopyPlacement>> host_placed;

  std::string reach_pool;
  bool reach_answer = false;
  auto start_chunk = [&](Chunk& ch) {
    const TimePoint t0 = Clock::now();
    BB_TRACE_SPAN("put.start_chunk", ch.end - ch.begin);
    std::vector<PutStartItem> items;
    items.reserve(ch.end - ch.begin);
    for (size_t i = ch.begin; i < ch.end; ++i) items.push_back(PutStartItem{keys[i], sizes[i], cfg});
    ch.placed = keystone_->batch_put_start(items);  // one control-plane round trip per chunk
    rpc_us_total += us_since(t0);
    metrics_.observe("phase_put_start_us", us_since(t0));
    // One descriptor per (object, shard): copy 0's placement plus the same shard of every other
    // copy as extra destinations, so the kernel reads the source once and fans out.
    for (size_t i = ch.begin; i < ch.end; ++i) {
      const auto& pr = ch.placed[i - ch.begin];
      if (!pr.ok()) {
        out[i] = pr.error();
        continue;
      }
      out[i] = ErrorCode::OK;
      const auto& copies = pr.value();
      if (copies.empty()) continue;
      // placements on host tiers (DRAM / CXL / NVMe): stage through host memory and use the data servers
      bool on_fabric = true;
      for (const auto& c : copies)
        for (const auto& sh : c.shards) {
          // a batch lands on a handful of pools: ask the transport once per run of shards on the same pool
          if (reach_pool.empty() || reach_pool != sh.pool_id || !reach_answer) {
            reach_answer = device_->can_reach(sh);
            reach_pool = sh.pool_id;
          }
          on_fabric &= reach_answer;
        }
      if (!on_fabric) {
        host_put.push_back(i);
        host_placed[i] = copies;
        continue;
      }
      bool same_layout = true;
      for (const auto& c : copies) same_layout &= c.shards.size() == copies[0].shards.size();
      if (same_layout) {
        uint64_t off = 0;
        for (size_t s = 0; s < copies[0].shards.size(); ++s) {
          DeviceShardOp op;
          op.item = i;
          op.copy = 0;
          op.shard = s;
          op.placement = &copies[0].shards[s];
          op.obj_offset = off;
          if (sv) op.segs = sv->segs + sv->first[i], op.nsegs = sv->count[i];
          for (size_t c = 1; c < copies.size(); ++c) op.replicas.push_back(&copies[c].shards[s]);
          ch.ops.push_back(std::move(op));
          off += copies[0].shards[s].length;
        }
      } else {
        for (size_t c = 0; c < copies.size(); ++c) {
          uint64_t o2 = 0;
          for (size_t s = 0; s < copies[c].shards.size(); ++s) {
            DeviceShardOp op;
            op.item = i;
            op.copy = c;
            op.shard = s;
            op.placement = &copies[c].shards[s];
            op.obj_offset = o2;
            if (sv) op.segs = sv->segs + sv->first[i], op.nsegs = sv->count[i];
            ch.ops.push_back(std::move(op));
            o2 += copies[c].shards[s].length;
          }
        }
      }
    }
    const TimePoint t1 = Clock::now();
    auto t = device_->submit_put(ch.ops, dev_ptrs, cfg.checksum, stream);
    metrics_.observe("phase_put_submit_us", us_since(t1));
    if (t.ok()) {
      ch.ticket = t.value();
      ch.submitted = true;
    } else {
      ch.submit_error = t.error();
    }
  };

  auto finish_chunk = [&](Chunk& ch) {
    BB_TRACE_SPAN("finish_chunk", ch.end - ch.begin);
    std::vector<uint64_t> digests;
    ErrorCode ec = ch.submit_error;
    const TimePoint t1 = Clock::now();
    if (ch.submitted) ec = device_->wait_put(ch.ticket, &digests);
    metrics_.observe("phase_put_wait_us", us_since(t1));
    const TimePoint t2 = Clock::now();
    std::vector<ObjectKey> done_keys, cancel_keys;
    std::vector<ShardChecksums> done_sums;
    std::vector<size_t> done_idx;
    if (ec != ErrorCode::OK) {
      for (size_t i = ch.begin; i < ch.end; ++i)
        if (ch.placed[i - ch.begin].ok()) {
          out[i] = ec;
          cancel_keys.push_back(keys[i]);
        }
    } else {
      std::vector<ShardChecksums> sums(ch.end - ch.begin);
      for (size_t i = ch.begin; i < ch.end; ++i) {
        const auto& pr = ch.placed[i - ch.begin];
        if (!pr.ok()) continue;
        auto& sm = sums[i - ch.begin];
        sm.resize(pr.value().size());
        for (size_t c = 0; c < sm.size(); ++c) sm[c].assign(pr.value()[c].shards.size(), 0);
      }
      for (size_t k = 0; k < ch.ops.size(); ++k) {
        const auto& op = ch.ops[k];
        auto& sm = sums[op.item - ch.begin];
        sm[op.copy][op.shard] = digests[k];
        for (size_t r = 0; r < op.replicas.size(); ++r) sm[r + 1][op.shard] = digests[k];
      }
      for (size_t i = ch.begin; i < ch.end; ++i)
        if (ch.placed[i - ch.begin].ok() && !host_placed.count(i)) {
          done_keys.push_back(keys[i]);
          done_sums.push_back(std::move(sums[i - ch.begin]));
          done_idx.push_back(i);
        }
    }
    if (!cancel_keys.empty()) keystone_->batch_put_cancel(cancel_keys);
    if (!done_keys.empty()) {
      auto ecs = keystone_->batch_put_complete(done_keys, done_sums);
      for (size_t k = 0; k < done_idx.size(); ++k) out[done_idx[k]] = ecs[k];
    }
    rpc_us_total += us_since(t2);
    metrics_.observe("phase_put_complete_us", us_since(t2));
  };

  const size_t depth = std::max<size_t>(1, std::min<size_t>(2, device_->max_in_flight()));
  size_t finished = 0;
  for (size_t c = 0; c < chunks.size(); ++c) {
    while (c - finished >= depth) finish_chunk(chunks[finished++]);  // at most `depth` chunks in flight
    chunks[c].begin = plan[c].first;
    chunks[c].end = plan[c].second;
    start_chunk(chunks[c]);
  }
  while (finished < chunks.size()) finish_chunk(chunks[finished++]);
  // host-tier placements: D2H into a staging buffer, then the TCP data path (checksums on the CPU)
  for (size_t i : host_put) {
    std::vector<uint8_t> stage(sizes[i]);
    ErrorCode ec = ErrorCode::OK;
    if (sv) {  // gather: one D2H per segment
      uint64_t pos = 0;
      for (size_t k = 0; k < sv->count[i] && ec == ErrorCode::OK; ++k) {
        const DeviceSegment& sg = sv->segs[sv->first[i] + k];
        ec = device_->copy_d2h(stage.data() + pos, reinterpret_cast<const void*>(sg.ptr), sg.len, stream);
        pos += sg.len;
      }
    } else {
      ec = device_->copy_d2h(stage.data(), dev_ptrs[i], sizes[i], stream);
    }
    ShardChecksums sums;
    if (ec == ErrorCode::OK) ec = transfer_put(host_placed[i], stage.data(), cfg.checksum, &sums);
    if (ec == ErrorCode::OK) ec = keystone_->put_complete(keys[i], sums);
    else keystone_->put_cancel(keys[i]);
    out[i] = ec;
    metrics_.inc("device_put_host_staged_total");
  }
  if (!keys.empty()) ewma_update(put_rpc_us_per_obj_, rpc_us_total / static_cast<double>(keys.size()));
  metrics_.inc("device_put_batches_total");
  metrics_.observe("device_put_batch_latency_us", us_since(t_all));
  return out;
}

std::vector<ErrorCode> BlackbirdClient::batch_get_device(const std::vector<ObjectKey>& keys, const std::vector<void*>& dev_ptrs,
                                                         const std::vector<size_t>& capacity, void* stream,
                                                         std::vector<size_t>* out_sizes) {
  return get_device_impl(keys, dev_ptrs, capacity, nullptr, stream, out_sizes);
}

std::vector<ErrorCode> BlackbirdClient::batch_get_device_scatter(const std::vector<ObjectKey>& keys, const std::vector<DeviceSegment>& segs,
                                                                 const std::vector<uint32_t>& seg_counts, void* stream) {
  std::vector<ErrorCode> out(keys.size(), ErrorCode::INVALID_PARAMETERS);
  if (!keystone_) return std::vector<ErrorCode>(keys.size(), ErrorCode::CLIENT_DISCONNECTED);
  if (!device_) return std::vector<ErrorCode>(keys.size(), ErrorCode::NOT_IMPLEMENTED);
  std::vector<size_t> first, total;
  if (seg_counts.size() != keys.size() || !index_segments(segs, seg_counts, &first, &out, &total))
    return std::vector<ErrorCode>(keys.size(), ErrorCode::INVALID_PARAMETERS);
  SegView sv;
  sv.segs = segs.data();
  std::vector<ObjectKey> vkeys;
  std::vector<size_t> idx, caps;
  for (size_t i = 0; i < keys.size(); ++i) {
    if (out[i] != ErrorCode::OK) continue;
    idx.push_back(i), vkeys.push_back(keys[i]), caps.push_back(total[i]);
    sv.first.push_back(first[i]), sv.count.push_back(seg_counts[i]);
  }
  if (idx.empty()) return out;
  auto r = get_device_impl(vkeys, std::vector<void*>(idx.size(), nullptr), caps, &sv, stream, nullptr);
  for (size_t k = 0; k < idx.size(); ++k) out[idx[k]] = r[k];
  return out;
}

std::vector<ErrorCode> BlackbirdClient::get_device_impl(const std::vector<ObjectKey>& keys, const std::vector<void*>& dev_ptrs,
                                                        const std::vector<size_t>& capacity, const SegView* sv, void* stream,
                                                        std::vector<size_t>* out_sizes) {
  std::vector<ErrorCode> out(keys.size(), ErrorCode::INVALID_PARAMETERS);
  if (!keystone_) return std::vector<ErrorCode>(keys.size(), ErrorCode::CLIENT_DISCONNECTED);
  if (!device_) return std::vector<ErrorCode>(keys.size(), ErrorCode::NOT_IMPLEMENTED);
  if (dev_ptrs.size() != keys.size() || capacity.size() != keys.size()) return out;
  const TimePoint t_all = Clock::now();
  BB_TRACE_SPAN("batch_get_device", keys.size());
  if (out_sizes) out_sizes->assign(keys.size(), 0);
  std::vector<Result<std::vector<CopyPlacement>>> placed(keys.size(), Result<std::vector<CopyPlacement>>(ErrorCode::INTERNAL_ERROR));
  std::vector<size_t> copy_choice(keys.size(), 0);
  std::vector<bool> pending(keys.size(), false);

  auto build_ops = [&](size_t begin, size_t end, std::vector<DeviceShardOp>& ops) {
    for (size_t i = begin; i < end; ++i) {
      if (!pending[i]) continue;
      const auto& copies = placed[i].value();
      const auto& copy = copies[copy_choice[i] % copies.size()];
      uint64_t off = 0;
      for (size_t s = 0; s < copy.shards.size(); ++s) {
        DeviceShardOp op;
        op.item = i;
        op.copy = copy_choice[i] % copies.size();
        op.shard = s;
        op.placement = &copy.shards[s];
        op.obj_offset = off;
        if (sv) op.segs = sv->segs + sv->first[i], op.nsegs = sv->count[i];
        ops.push_back(std::move(op));
        off += copy.shards[s].length;
      }
    }
  };
  auto apply_status = [&](const std::vector<DeviceShardOp>& ops, const std::vector<uint32_t>& status, std::vector<size_t>* retry) {
    std::vector<bool> bad(keys.size(), false), seen(keys.size(), false);
    for (size_t k = 0; k < ops.size(); ++k) {
      seen[ops[k].item] = true;
      if (status[k] != 0) bad[ops[k].item] = true;
    }
    for (size_t i = 0; i < keys.size(); ++i) {
      if (!seen[i] || !pending[i]) continue;
      if (!bad[i]) {
        out[i] = ErrorCode::OK;
        pending[i] = false;
      } else {
        metrics_.inc("checksum_mismatch_total");
        ++copy_choice[i];  // fail over to the next replica
        if (retry) retry->push_back(i);
      }
    }
  };

  // ---- first attempt: chunks pipelined against the get_workers round trips
  struct Chunk {
    size_t begin = 0, end = 0;
    std::vector<DeviceShardOp> ops;
    uint64_t ticket = 0;
    bool submitted = false;
    ErrorCode err = ErrorCode::OK;
  };
  auto plan = plan_chunks(capacity, get_rpc_us_per_obj_.load(std::memory_order_relaxed));
  if (sv) plan = cap_chunk_segments(plan, sv->count);
  double rpc_us_total = 0;
  std::vector<Chunk> chunks(plan.size());
  std::vector<size_t> retry;
  // A batch mostly reads from a handful of pools: remember the transport's answer for the last pool asked about instead of
  // taking its lock and looking the pool id up once per shard, and count per-object events locally (a named counter is a
  // map lookup under a mutex).
  const std::string* local_pool = nullptr;
  bool local_answer = false;
  auto pool_is_local = [&](const ShardPlacement& sh) {
    if (!local_pool || *local_pool != sh.pool_id) {
      local_answer = device_->is_local(sh);
      local_pool = &sh.pool_id;
    }
    return local_answer;
  };
  std::string reach_pool;
  bool reach_answer = false;
  auto pool_reachable = [&](const ShardPlacement& sh) {
    if (reach_pool.empty() || reach_pool != sh.pool_id || !reach_answer) {
      reach_answer = device_->can_reach(sh);
      reach_pool = sh.pool_id;
    }
    return reach_answer;
  };
  uint64_t n_local = 0, n_dram_direct = 0;
  auto start_chunk = [&](Chunk& ch) {
    const TimePoint t0 = Clock::now();
    local_pool = nullptr;  // the cached pointer refers into the previous chunk's placements
    const bool whole = ch.begin == 0 && ch.end == keys.size();
    std::vector<ObjectKey> part;
    if (!whole) part.assign(keys.begin() + static_cast<std::ptrdiff_t>(ch.begin), keys.begin() + static_cast<std::ptrdiff_t>(ch.end));
    const std::vector<ObjectKey>& ck = whole ? keys : part;
    auto res = keystone_->batch_get_workers(ck);
    rpc_us_total += us_since(t0);
    metrics_.observe("phase_get_workers_us", us_since(t0));
    for (size_t i = ch.begin; i < ch.end; ++i) {
      placed[i] = std::move(res[i - ch.begin]);
      if (!placed[i].ok()) {
        out[i] = placed[i].error();
        continue;
      }
      if (placed[i].value().empty()) {
        out[i] = ErrorCode::NO_COMPLETE_WORKER;
        continue;
      }
      size_t size = 0;
      for (const auto& s : placed[i].value()[0].shards) size += s.length;
      if (out_sizes) (*out_sizes)[i] = size;
      if (sv && size != capacity[i]) {  // a scatter list must cover the object exactly
        out[i] = ErrorCode::INVALID_PARAMETERS;
        continue;
      }
      if (size > capacity[i]) {
        out[i] = ErrorCode::BUFFER_OVERFLOW;
        continue;
      }
      // replica choice: one that lives on this client's own GPU (HBM speed, no NVLink), else a replica that is
      // fully reachable over the GPU fabric (readers spread over the replicas), else stage through the host
      const auto& copies = placed[i].value();
      // (the spread over replicas only matters when there is more than one; thousands of single-copy objects skip the hash)
      const size_t start = copies.size() > 1 ? std::hash<std::string>{}(opts_.node_id + keys[i]) % copies.size() : 0;
      bool found = false;
      for (size_t k = 0; k < copies.size() && !found; ++k) {
        bool local = !copies[k].shards.empty();
        for (const auto& sh : copies[k].shards) local &= pool_is_local(sh);
        if (local) {
          copy_choice[i] = k;
          found = true;
          ++n_local;
        }
      }
      // HBM replicas first (NVLink), then replicas in mapped DRAM pools (PCIe)
      for (int pass = 0; pass < 2 && !found; ++pass) {
        for (size_t k = 0; k < copies.size() && !found; ++k) {
          const auto& c = copies[(start + k) % copies.size()];
          bool ok = !c.shards.empty();
          for (const auto& sh : c.shards) ok = ok && (pass == 1 || sh.storage_class == StorageClass::RAM_GPU) && pool_reachable(sh);
          if (ok) {
            copy_choice[i] = (start + k) % copies.size();
            found = true;
            if (pass == 1) ++n_dram_direct;
          }
        }
      }
      if (!found) {
        std::vector<uint8_t> stage(size);
        ErrorCode ec = transfer_get(copies, stage.data(), size);  // data servers + CPU checksum + replica fail-over
        if (ec == ErrorCode::OK && sv) {  // scatter: one H2D per segment
          uint64_t pos = 0;
          for (size_t k = 0; k < sv->count[i] && ec == ErrorCode::OK; ++k) {
            const DeviceSegment& sg = sv->segs[sv->first[i] + k];
            ec = device_->copy_h2d(reinterpret_cast<void*>(sg.ptr), stage.data() + pos, sg.len, stream);
            pos += sg.len;
          }
        } else if (ec == ErrorCode::OK) {
          ec = device_->copy_h2d(dev_ptrs[i], stage.data(), size, stream);
        }
        out[i] = ec;
        metrics_.inc("device_get_host_staged_total");
        continue;
      }
      pending[i] = true;
    }
    build_ops(ch.begin, ch.end, ch.ops);
    if (ch.ops.empty()) return;
    const TimePoint t1 = Clock::now();
    auto t = device_->submit_get(ch.ops, dev_ptrs, stream);
    metrics_.observe("phase_get_submit_us", us_since(t1));
    if (t.ok()) {
      ch.ticket = t.value();
      ch.submitted = true;
    } else {
      ch.err = t.error();
    }
  };
  auto finish_chunk = [&](Chunk& ch) {
    BB_TRACE_SPAN("finish_chunk", ch.end - ch.begin);
    if (ch.ops.empty()) return;
    std::vector<uint32_t> status;
    ErrorCode ec = ch.err;
    const TimePoint t1 = Clock::now();
    if (ch.submitted) ec = device_->wait_get(ch.ticket, &status);
    metrics_.observe("phase_get_wait_us", us_since(t1));
    if (ec != ErrorCode::OK) {
      for (size_t i = ch.begin; i < ch.end; ++i)
        if (pending[i]) {
          out[i] = ec;
          pending[i] = false;
        }
      return;
    }
    apply_status(ch.ops, status, &retry);
  };
  const size_t depth = std::max<size_t>(1, std::min<size_t>(2, device_->max_in_flight()));
  size_t finished = 0;
  for (size_t c = 0; c < chunks.size(); ++c) {
    while (c - finished >= depth) finish_chunk(chunks[finished++]);  // at most `depth` chunks in flight
    chunks[c].begin = plan[c].first;
    chunks[c].end = plan[c].second;
    start_chunk(chunks[c]);
  }
  while (finished < chunks.size()) finish_chunk(chunks[finished++]);

  // ---- replica fail-over for objects whose digest did not verify
  for (size_t attempt = 1; attempt < 4 && !retry.empty(); ++attempt) {
    std::vector<size_t> still;
    std::vector<DeviceShardOp> ops;
    for (size_t i : retry) {
      if (attempt >= placed[i].value().size()) {
        out[i] = ErrorCode::CHECKSUM_MISMATCH;
        pending[i] = false;
      }
    }
    build_ops(0, keys.size(), ops);
    if (ops.empty()) break;
    metrics_.inc("replica_failover_total");
    std::vector<uint32_t> status;
    ErrorCode ec = device_->get_shards(ops, dev_ptrs, ChecksumAlgo::NONE, stream, &status);
    if (ec != ErrorCode::OK) {
      for (size_t i = 0; i < keys.size(); ++i)
        if (pending[i]) {
          out[i] = ec;
          pending[i] = false;
        }
      break;
    }
    apply_status(ops, status, &still);
    retry.swap(still);
  }
  for (size_t i = 0; i < keys.size(); ++i)
    if (pending[i]) out[i] = ErrorCode::CHECKSUM_MISMATCH;
  if (n_local) metrics_.inc("device_get_local_replica_total", n_local);
  if (n_dram_direct) metrics_.inc("device_get_dram_direct_total", n_dram_direct);
  // ---- a mismatch can also mean that the Keystone moved the object under us (tier move, compaction, repair): the
  // extents we read were freed and re-used.  Objects whose placements changed since we fetched them get one more pass.
  static thread_local int refresh_depth = 0;
  if (refresh_depth < 2) {
    std::vector<size_t> bad;
    for (size_t i = 0; i < keys.size(); ++i)
      if (out[i] == ErrorCode::CHECKSUM_MISMATCH && placed[i].ok()) bad.push_back(i);
    if (!bad.empty()) {
      std::vector<ObjectKey> bkeys;
      for (size_t i : bad) bkeys.push_back(keys[i]);
      auto again = keystone_->batch_get_workers(bkeys);
      std::vector<ObjectKey> rkeys;
      std::vector<void*> rptrs;
      std::vector<size_t> rcaps, ridx;
      SegView rsv;
      if (sv) rsv.segs = sv->segs;
      for (size_t k = 0; k < bad.size(); ++k) {
        const size_t i = bad[k];
        if (!again[k].ok()) {
          out[i] = again[k].error();  // removed (or being re-written) meanwhile: that is the answer
        } else if (!(again[k].value() == placed[i].value()) || refresh_depth == 0) {
          // changed placements, or (once) the same ones: a remove + re-put can land on the very same extent (first fit)
          // and be read half-written
          rkeys.push_back(keys[i]), rptrs.push_back(dev_ptrs[i]), rcaps.push_back(capacity[i]), ridx.push_back(i);
          if (sv) rsv.first.push_back(sv->first[i]), rsv.count.push_back(sv->count[i]);
        }
      }
      if (!rkeys.empty()) {
        metrics_.inc("get_placement_refresh_total", rkeys.size());
        std::vector<size_t> rsizes;
        ++refresh_depth;
        auto recs = get_device_impl(rkeys, rptrs, rcaps, sv ? &rsv : nullptr, stream, &rsizes);
        --refresh_depth;
        for (size_t k = 0; k < ridx.size(); ++k) {
          out[ridx[k]] = recs[k];
          if (out_sizes && k < rsizes.size()) (*out_sizes)[ridx[k]] = rsizes[k];
        }
      }
    }
  }
  if (!keys.empty()) ewma_update(get_rpc_us_per_obj_, rpc_us_total / static_cast<double>(keys.size()));
  metrics_.inc("device_get_batches_total");
  metrics_.observe("device_get_batch_latency_us", us_since(t_all));
  return out;
}

// ================================================================ HostLoopbackTransport (CPU stand-in for the GPU fabric)
bool HostLoopbackTransport::can_reach(const ShardPlacement& s) const {
  if (s.storage_class == StorageClass::RAM_GPU) return false;
  return reach_disk_ || !is_disk_class(s.storage_class);
}

ErrorCode HostLoopbackTransport::put_shards(const std::vector<DeviceShardOp>& ops, const std::vector<const void*>& dev_ptrs, ChecksumAlgo algo,
                                            void*, std::vector<uint64_t>* digests) {
  ++launches_;  // one "launch" per batch, like the fused kernel
  if (digests) digests->assign(ops.size(), 0);
  std::vector<uint8_t> gathered;
  for (size_t k = 0; k < ops.size(); ++k) {
    const DeviceShardOp& op = ops[k];
    const auto* src = static_cast<const uint8_t*>(dev_ptrs[op.item]) + op.obj_offset;
    if (op.segs) {  // gather this shard's slice of the segment list
      gathered.resize(op.placement->length);
      BB_TRY(copy_segments(op, gathered.data(), true));
      src = gathered.data();
    }
    uint64_t d = 0;
    ErrorCode ec = io_->write_shard(*op.placement, src, &d, algo);
    for (size_t r = 0; r < op.replicas.size() && ec == ErrorCode::OK; ++r) ec = io_->write_shard(*op.replicas[r], src, nullptr, ChecksumAlgo::NONE);
    if (ec != ErrorCode::OK) return ec;
    if (digests) (*digests)[k] = d;
  }
  return ErrorCode::OK;
}

ErrorCode HostLoopbackTransport::get_shards(const std::vector<DeviceShardOp>& ops, const std::vector<void*>& dev_ptrs, ChecksumAlgo, void*,
                                            std::vector<uint32_t>* status) {
  ++launches_;
  if (status) status->assign(ops.size(), 0);
  std::vector<uint8_t> stage;
  for (size_t k = 0; k < ops.size(); ++k) {
    const DeviceShardOp& op = ops[k];
    auto* dst = static_cast<uint8_t*>(dev_ptrs[op.item]) + op.obj_offset;
    if (op.segs) {
      stage.resize(op.placement->length);
      dst = stage.data();
    }
    const ErrorCode ec = io_->read_shard(*op.placement, dst, op.placement->checksum_algo);
    if (ec == ErrorCode::CHECKSUM_MISMATCH) {
      if (status) (*status)[k] = 1;  // reported per shard, like the kernel's verify flag
      if (op.segs) BB_TRY(copy_segments(op, stage.data(), false));  // the kernel stores what it read, verified or not
    } else if (ec != ErrorCode::OK) {
      return ec;
    } else if (op.segs) {
      BB_TRY(copy_segments(op, stage.data(), false));  // scatter
    }
  }
  return ErrorCode::OK;
}

ErrorCode HostLoopbackTransport::copy_segments(const DeviceShardOp& op, uint8_t* buf, bool gather) {
  size_t k = 0;
  uint64_t skip = 0, left = op.placement->length;
  if (left == 0) return ErrorCode::OK;
  if (!segment_slice(op.segs, op.nsegs, op.obj_offset, &k, &skip)) return ErrorCode::INVALID_ARGUMENT;
  for (; k < op.nsegs && left; ++k, skip = 0) {
    const uint64_t n = std::min<uint64_t>(op.segs[k].len - skip, left);
    auto* seg = reinterpret_cast<uint8_t*>(op.segs[k].ptr) + skip;
    if (gather) std::memcpy(buf, seg, n);
    else std::memcpy(seg, buf, n);
    buf += n, left -= n;
  }
  return left ? ErrorCode::INVALID_ARGUMENT : ErrorCode::OK;
}

ErrorCode HostLoopbackTransport::put_fp8(const std::vector<DeviceFp8Op>& ops, void*, std::vector<uint64_t>* digests) {
  ++launches_;
  if (digests) digests->assign(ops.size(), 0);
  for (size_t k = 0; k < ops.size(); ++k) {
    const DeviceFp8Op& op = ops[k];
    std::vector<uint8_t> packed(mxfp8::packed_bytes(op.n_elems));
    mxfp8::pack_bf16(static_cast<const uint16_t*>(op.wide), op.n_elems, packed.data());
    uint64_t d = 0;
    ErrorCode ec = io_->write_shard(*op.placement, packed.data(), &d, ChecksumAlgo::BBH64);
    for (size_t r = 0; r < op.replicas.size() && ec == ErrorCode::OK; ++r) ec = io_->write_shard(*op.replicas[r], packed.data(), nullptr, ChecksumAlgo::NONE);
    if (ec != ErrorCode::OK) return ec;
    if (digests) (*digests)[k] = d;
  }
  return ErrorCode::OK;
}

ErrorCode HostLoopbackTransport::get_fp8(const std::vector<DeviceFp8Op>& ops, void*, std::vector<uint32_t>* status) {
  ++launches_;
  if (status) status->assign(ops.size(), 0);
  for (size_t k = 0; k < ops.size(); ++k) {
    const DeviceFp8Op& op = ops[k];
    std::vector<uint8_t> packed(mxfp8::packed_bytes(op.n_elems));
    const ErrorCode ec = io_->read_shard(*op.placement, packed.data(), ChecksumAlgo::BBH64);
    if (ec == ErrorCode::CHECKSUM_MISMATCH) {
      if (status) (*status)[k] = 1;
      continue;
    }
    if (ec != ErrorCode::OK) return ec;
    mxfp8::unpack_bf16(packed.data(), op.n_elems, static_cast<uint16_t*>(op.wide));
  }
  return ErrorCode::OK;
}

}  // namespace bb::client
