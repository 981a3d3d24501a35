#include "common/trace.h"
#include "fabric/gpu_fabric.h"

#include <cuda.h>
#include <cuda_runtime.h>

#include <cstring>

#include "common/log.h"

namespace bb::gpu {

namespace drv {
// cuMemGetAddressRange resolved at runtime (the module must import on a CPU-only box: no libcuda link dependency).
bool get_address_range(const void* p, CUdeviceptr* base, size_t* size) {
  static auto fn = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
      cudaGetLastError();
      f = nullptr;
    }
    return reinterpret_cast<CUresult (*)(CUdeviceptr*, size_t*, CUdeviceptr)>(f);
  }();
  if (!fn) return false;
  if (fn(base, size, reinterpret_cast<CUdeviceptr>(p)) != CUDA_SUCCESS) return false;
  // the range is that of the allocation containing p; what is left of it from p on:
  const size_t skip = reinterpret_cast<CUdeviceptr>(p) - *base;
  *size = *size > skip ? *size - skip : 0;
  return true;
}
}  // namespace drv

namespace {
struct LocalSlab {
  int device;
  void* base;
  uint64_t size;
};
std::mutex g_local_mu;
std::map<std::string, LocalSlab> g_local;

bool cuda_ok(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return true;
  BB_LOG(ERROR) << "CUDA error in " << what << ": " << cudaGetErrorString(e);
  cudaGetLastError();
  return false;
}
}  // namespace

void register_local_slab(const std::string& pool_id, int device, void* base, uint64_t size) {
  std::lock_guard<std::mutex> lk(g_local_mu);
  g_local[pool_id] = LocalSlab{device, base, size};
}
void unregister_local_slab(const std::string& pool_id) {
  std::lock_guard<std::mutex> lk(g_local_mu);
  g_local.erase(pool_id);
}

// ================================================================ GpuSlabBackend
GpuSlabBackend::GpuSlabBackend(uint64_t capacity, worker::BackendOptions opts)
    : StorageBackend(StorageClass::RAM_GPU, capacity, std::move(opts)) {}
GpuSlabBackend::~GpuSlabBackend() { shutdown(); }

ErrorCode GpuSlabBackend::initialize() {
  if (initialized_) return ErrorCode::OK;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || opts_.gpu_device_id >= n) {
    cudaGetLastError();
    return ErrorCode::INITIALIZATION_FAILED;
  }
  if (!cuda_ok(cudaSetDevice(opts_.gpu_device_id), "cudaSetDevice")) return ErrorCode::FABRIC_ERROR;
  void* p = nullptr;
  if (!cuda_ok(cudaMalloc(&p, capacity_), "cudaMalloc(slab)")) return ErrorCode::OUT_OF_MEMORY;
  base_ = static_cast<uint8_t*>(p);
  cudaIpcMemHandle_t h;
  if (cuda_ok(cudaIpcGetMemHandle(&h, p), "cudaIpcGetMemHandle")) {
    std::vector<uint8_t> raw(sizeof h);
    std::memcpy(raw.data(), &h, sizeof h);
    handle_hex_ = bytes_to_hex(raw);
  }
  cudaStream_t st;
  if (cuda_ok(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking), "cudaStreamCreate")) stream_ = st;
  rkey_ = reinterpret_cast<uint64_t>(p) >> 8;
  init_allocator();
  register_local_slab(pool_id_, opts_.gpu_device_id, base_, capacity_);
  // engine of the tier-move / repair paths: created now, because allocating it later would synchronise the device
  // in the middle of somebody's collective
  if (auto e = XferEngine::create(opts_.gpu_device_id, 64, 1); e.ok()) move_engine_ = std::move(e.value());
  initialized_ = true;
  return ErrorCode::OK;
}

void GpuSlabBackend::shutdown() {
  if (!base_) return;

  unregister_local_slab(pool_id_);
  cudaSetDevice(opts_.gpu_device_id);
  if (stream_) cudaStreamDestroy(static_cast<cudaStream_t>(stream_));
  cudaFree(base_);
  base_ = nullptr;
  stream_ = nullptr;
  initialized_ = false;
}

ErrorCode GpuSlabBackend::write(uint64_t offset, const void* data, uint64_t len) {
  BB_TRY(check_range(offset, len));
  cudaStream_t st = static_cast<cudaStream_t>(stream_);
  if (!cuda_ok(cudaSetDevice(opts_.gpu_device_id), "cudaSetDevice") ||
      !cuda_ok(cudaMemcpyAsync(base_ + offset, data, len, cudaMemcpyHostToDevice, st), "H2D") ||
      !cuda_ok(cudaStreamSynchronize(st), "sync"))
    return ErrorCode::FABRIC_ERROR;
  bytes_written_ += len;
  return ErrorCode::OK;
}

ErrorCode GpuSlabBackend::read(uint64_t offset, void* data, uint64_t len) {
  BB_TRY(check_range(offset, len));
  cudaStream_t st = static_cast<cudaStream_t>(stream_);
  if (!cuda_ok(cudaSetDevice(opts_.gpu_device_id), "cudaSetDevice") ||
      !cuda_ok(cudaMemcpyAsync(data, base_ + offset, len, cudaMemcpyDeviceToHost, st), "D2H") ||
      !cuda_ok(cudaStreamSynchronize(st), "sync"))
    return ErrorCode::FABRIC_ERROR;
  bytes_read_ += len;
  return ErrorCode::OK;
}

// Peer slabs are mapped once per process and device: the client-side fabric and the worker-side repair path
// (pull_from_peer) share the mapping, and nothing is unmapped before the process exits (a mapping may be in use by
// a kernel of either side).  Opening is a device-synchronising driver call, so it must not happen lazily on a hot path.
static std::mutex g_ipc_mu;
static std::map<std::pair<int, std::string>, void*> g_ipc_mapped;  // (device, handle bytes) -> base
static void* ipc_map_peer_slab(int device, const cudaIpcMemHandle_t& h, cudaError_t* err) {
  const std::string key(reinterpret_cast<const char*>(&h), sizeof h);
  std::lock_guard<std::mutex> lk(g_ipc_mu);
  auto it = g_ipc_mapped.find({device, key});
  if (it != g_ipc_mapped.end()) return it->second;
  void* ptr = nullptr;
  cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
  if (err) *err = e;
  if (e != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  g_ipc_mapped[{device, key}] = ptr;
  return ptr;
}

ErrorCode GpuSlabBackend::device_copy(worker::StorageBackend& peer, bool to_peer, uint64_t my_off, uint64_t peer_off, uint64_t len,
                                      ChecksumAlgo algo, uint64_t* digest) {
  if (!base_ || !peer.cuda_accessible()) return ErrorCode::NOT_IMPLEMENTED;
  BB_TRY(check_range(my_off, len));
  auto* theirs = static_cast<uint8_t*>(peer.direct_ptr(peer_off));
  const uint64_t peer_cap = peer.get_total_capacity();
  if (!theirs || len > peer_cap || peer_off > peer_cap - len) return ErrorCode::MEMORY_ACCESS_ERROR;  // overflow safe
  uint8_t* mine = base_ + my_off;
  if ((reinterpret_cast<uintptr_t>(mine) | reinterpret_cast<uintptr_t>(theirs)) & 15) return ErrorCode::NOT_IMPLEMENTED;  // staged path handles it
  std::lock_guard<std::mutex> lk(move_mu_);
  if (!cuda_ok(cudaSetDevice(opts_.gpu_device_id), "cudaSetDevice")) return ErrorCode::FABRIC_ERROR;
  if (!move_engine_) {
    auto e = XferEngine::create(opts_.gpu_device_id, 64, 1);
    if (!e.ok()) return e.error();
    move_engine_ = std::move(e.value());
  }
  XferItem it;
  it.src = to_peer ? mine : theirs;
  it.dst[0] = to_peer ? theirs : mine;
  it.ndst = 1;
  it.nbytes = len;
  XferResult res;
  ErrorCode ec = move_engine_->run({it}, algo, stream_, &res);
  if (ec != ErrorCode::OK) return ec;
  if (digest) *digest = res.digest.empty() ? 0 : res.digest[0];
  (to_peer ? bytes_read_ : bytes_written_) += len;
  ++device_copies_;
  return ErrorCode::OK;
}

ErrorCode GpuSlabBackend::pull_from_peer(const std::vector<uint8_t>& peer_key, uint64_t peer_off, uint64_t my_off, uint64_t len,
                                         ChecksumAlgo algo, uint64_t* digest) {
  if (!base_ || peer_key.size() != sizeof(cudaIpcMemHandle_t)) return ErrorCode::NOT_IMPLEMENTED;
  BB_TRY(check_range(my_off, len));
  std::lock_guard<std::mutex> lk(move_mu_);
  if (!cuda_ok(cudaSetDevice(opts_.gpu_device_id), "cudaSetDevice")) return ErrorCode::FABRIC_ERROR;
  cudaIpcMemHandle_t h;
  std::memcpy(&h, peer_key.data(), sizeof h);
  cudaError_t e = cudaSuccess;
  void* peer_base = ipc_map_peer_slab(opts_.gpu_device_id, h, &e);
  if (!peer_base) {  // same-process slab, no peer access, stale handle: the caller relays through the data servers
    BB_VLOG(1) << "pull_from_peer: cannot map the peer slab (" << cudaGetErrorString(e) << ")";
    return ErrorCode::NOT_IMPLEMENTED;
  }
  // The mapping covers the peer's whole cudaMalloc allocation: bound the read by its real extent, so a bad
  // (peer_off, len) from the wire cannot make the copy kernel read past the mapped slab.
  {
    CUdeviceptr range_base = 0;
    size_t range_size = 0;
    if (!drv::get_address_range(peer_base, &range_base, &range_size) ||
        len > range_size || peer_off > range_size - len)
      return ErrorCode::MEMORY_ACCESS_ERROR;
  }
  uint8_t* theirs = static_cast<uint8_t*>(peer_base) + peer_off;
  uint8_t* mine = base_ + my_off;
  if ((reinterpret_cast<uintptr_t>(mine) | reinterpret_cast<uintptr_t>(theirs)) & 15) return ErrorCode::NOT_IMPLEMENTED;
  if (!move_engine_) {
    auto e = XferEngine::create(opts_.gpu_device_id, 64, 1);
    if (!e.ok()) return e.error();
    move_engine_ = std::move(e.value());
  }
  XferItem item;
  item.src = theirs;
  item.dst[0] = mine;
  item.ndst = 1;
  item.nbytes = len;
  XferResult res;
  ErrorCode ec = move_engine_->run({item}, algo, stream_, &res);
  if (ec != ErrorCode::OK) return ec;
  if (digest) *digest = res.digest.empty() ? 0 : res.digest[0];
  bytes_written_ += len;
  ++device_copies_;
  return ErrorCode::OK;
}

void install_gpu_backend_factory() {
  worker::HostPinHooks hooks;
  hooks.pin = [](void* p, uint64_t n) {
    int cnt = 0;
    if (cudaGetDeviceCount(&cnt) != cudaSuccess || cnt == 0) {
      cudaGetLastError();
      return false;
    }
    // portable: usable from every device context of this process; the kernels address it through UVA
    cudaError_t e = cudaHostRegister(p, n, cudaHostRegisterPortable | cudaHostRegisterMapped);
    if (e != cudaSuccess) {
      BB_LOG(WARNING) << "cudaHostRegister(" << n << " B) failed: " << cudaGetErrorString(e);
      cudaGetLastError();
      return false;
    }
    return true;
  };
  hooks.unpin = [](void* p) {
    if (cudaHostUnregister(p) != cudaSuccess) cudaGetLastError();
  };
  worker::set_host_pin_hooks(std::move(hooks));
  worker::set_gpu_backend_factory([](uint64_t capacity, const worker::BackendOptions& o) -> std::unique_ptr<worker::StorageBackend> {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
      cudaGetLastError();
      return nullptr;
    }
    return std::make_unique<GpuSlabBackend>(capacity, o);
  });
}

// ================================================================ GpuFabric
Result<std::shared_ptr<GpuFabric>> GpuFabric::create(int device, std::shared_ptr<rpc::KeystoneApi> keystone) {
  std::shared_ptr<GpuFabric> f(new GpuFabric());
  f->device_ = device;
  f->keystone_ = std::move(keystone);
  auto e = XferEngine::create(device, 1u << 16, 4);
  if (!e.ok()) return e.error();
  f->engine_ = std::move(e.value());
  if (f->keystone_) f->refresh_pools();
  return f;
}

GpuFabric::~GpuFabric() {
  std::lock_guard<std::mutex> lk(mu_);
  cudaSetDevice(device_);
  for (auto& [id, m] : pools_) {
    // IPC mappings are process-wide (ipc_map_peer_slab) and stay mapped; shared DRAM pools are ours
    if (m.host_mapped && m.base) {
      if (cudaHostUnregister(m.base) != cudaSuccess) cudaGetLastError();
      worker::unmap_shared_pool(m.base, m.size);
    }
  }
}

size_t GpuFabric::mapped_host_pools() const {
  std::lock_guard<std::mutex> lk(mu_);
  size_t n = 0;
  for (const auto& [id, m] : pools_) n += m.host ? 1 : 0;
  return n;
}

// DRAM-tier pools: in-process pinned pools are used as they are; pools of other worker processes on this host are
// memfd-backed ("file:/proc/<pid>/fd/<n>" registration key) and get mapped + cudaHostRegister'ed here, once, on the
// first shard that needs them.  Everything else (other host, private mapping) stays on the data-server path.
bool GpuFabric::ensure_host_pool(const std::string& pool_id) {
  for (int attempt = 0; attempt < 2; ++attempt) {
    HostCandidate cand;
    {
      std::lock_guard<std::mutex> lk(mu_);
      auto it = pools_.find(pool_id);
      if (it != pools_.end()) return it->second.host;
      if (host_unreachable_.count(pool_id)) return false;
      auto c = host_candidates_.find(pool_id);
      if (c == host_candidates_.end()) {
        if (attempt == 1) {
          host_unreachable_.insert(pool_id);
          return false;
        }
      } else {
        cand = c->second;
      }
    }
    if (cand.size == 0) {
      refresh_pools();  // a worker that joined after this fabric was created
      continue;
    }
    Mapping m;
    m.host = true;
    m.size = cand.size;
    m.remote_base = cand.remote_base;
    worker::LocalHostPool local;
    if (worker::find_local_host_pool(pool_id, &local) && local.size >= cand.size) {
      m.base = static_cast<uint8_t*>(local.base);  // pinned by the worker of this process
    } else if (auto raw = hex_to_bytes(cand.key_hex); raw) {
      m.key = *raw;
      void* p = worker::map_shared_pool(*raw, cand.size);
      if (p) {
        if (cuda_ok(cudaSetDevice(device_), "cudaSetDevice") &&
            cuda_ok(cudaHostRegister(p, cand.size, cudaHostRegisterPortable | cudaHostRegisterMapped), "cudaHostRegister(shared DRAM pool)")) {
          m.base = static_cast<uint8_t*>(p);
          m.host_mapped = true;
        } else {
          worker::unmap_shared_pool(p, cand.size);
        }
      }
    }
    std::lock_guard<std::mutex> lk(mu_);
    if (!m.base) {
      host_unreachable_.insert(pool_id);
      return false;
    }
    auto [it, fresh] = pools_.emplace(pool_id, m);
    if (!fresh && m.host_mapped) {  // lost a race with another thread: keep theirs
      if (cudaHostUnregister(m.base) != cudaSuccess) cudaGetLastError();
      worker::unmap_shared_pool(m.base, m.size);
    }
    BB_LOG(INFO) << "GPU " << device_ << ": DRAM pool " << pool_id << " (" << (cand.size >> 20) << " MiB) is reachable by the fused kernels ("
                 << (it->second.host_mapped ? "mapped from its worker's memfd" : "in-process pinned pool") << ")";
    return true;
  }
  return false;
}

size_t GpuFabric::mapped_pools() const {
  std::lock_guard<std::mutex> lk(mu_);
  return pools_.size();
}

ErrorCode GpuFabric::refresh_pools() {
  if (!keystone_) return ErrorCode::INVALID_STATE;
  auto pools = keystone_->get_memory_pools();
  if (!pools.ok()) return pools.error();
  if (!cuda_ok(cudaSetDevice(device_), "cudaSetDevice")) return ErrorCode::FABRIC_ERROR;
  std::lock_guard<std::mutex> lk(mu_);
  for (const auto& p : pools.value()) {
    if (p.storage_class == StorageClass::RAM_CPU) {
      if (!pools_.count(p.id)) host_candidates_[p.id] = HostCandidate{p.size, p.ucx_remote_addr ? p.ucx_remote_addr : p.base_addr, p.ucx_rkey_hex};
      continue;
    }
    if (p.storage_class != StorageClass::RAM_GPU || pools_.count(p.id)) continue;
    Mapping m;
    m.size = p.size;
    m.device = p.gpu_device_id;
    {
      std::lock_guard<std::mutex> l2(g_local_mu);
      auto it = g_local.find(p.id);
      if (it != g_local.end()) {
        m.base = static_cast<uint8_t*>(it->second.base);
        m.device = it->second.device;
        if (auto raw = hex_to_bytes(p.ucx_rkey_hex)) m.key = *raw;
      }
    }
    if (m.base) {
      if (m.device != device_) {
        int can = 0;
        cudaDeviceCanAccessPeer(&can, device_, m.device);
        if (!can) {
          BB_LOG(WARNING) << "GPU " << device_ << " cannot access peer " << m.device << "; pool " << p.id << " unreachable";
          continue;
        }
        cudaError_t e = cudaDeviceEnablePeerAccess(m.device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
          cuda_ok(e, "cudaDeviceEnablePeerAccess");
          continue;
        }
        cudaGetLastError();
      }
    } else {
      size_t grp = 0;
      int member = 0;
      if (NvlsArena::parse_pool_id(p.id, &grp, &member)) continue;  // VMM arena pools are mapped by NvlsArena, not by IPC
      auto raw = hex_to_bytes(p.ucx_rkey_hex);
      if (!raw || raw->size() != sizeof(cudaIpcMemHandle_t)) {
        BB_LOG(WARNING) << "pool " << p.id << " has no usable IPC handle";
        continue;
      }
      cudaIpcMemHandle_t h;
      std::memcpy(&h, raw->data(), sizeof h);
      cudaError_t ipc_err = cudaSuccess;
      void* ptr = ipc_map_peer_slab(device_, h, &ipc_err);
      if (!ptr) {
        cuda_ok(ipc_err, "cudaIpcOpenMemHandle");
        continue;
      }
      m.base = static_cast<uint8_t*>(ptr);
      m.ipc_opened = true;
      m.key = *raw;
    }
    pools_[p.id] = m;
  }
  return ErrorCode::OK;
}

void GpuFabric::drop_if_stale(const ShardPlacement& s) {
  if (s.endpoint.worker_key.empty()) return;
  std::lock_guard<std::mutex> lk(mu_);
  auto it = pools_.find(s.pool_id);
  if (it == pools_.end() || it->second.key.empty() || it->second.key == s.endpoint.worker_key) return;
  BB_LOG(WARNING) << "GPU " << device_ << ": pool " << s.pool_id << " was re-registered under a new key; dropping the stale mapping";
  if (it->second.host_mapped && it->second.base) {
    if (cudaHostUnregister(it->second.base) != cudaSuccess) cudaGetLastError();
    worker::unmap_shared_pool(it->second.base, it->second.size);
  }
  pools_.erase(it);
  host_candidates_.erase(s.pool_id);  // re-read the pool record (size / base / key) on the next use
  host_unreachable_.erase(s.pool_id);
  ++remaps_;
}

bool GpuFabric::can_reach(const ShardPlacement& s) const {
  const_cast<GpuFabric*>(this)->drop_if_stale(s);
  if (s.storage_class == StorageClass::RAM_CPU && std::holds_alternative<MemoryLocation>(s.location))
    return const_cast<GpuFabric*>(this)->ensure_host_pool(s.pool_id);
  if (s.storage_class != StorageClass::RAM_GPU) return false;
  size_t grp = 0;
  int member = 0;
  if (arena_ && NvlsArena::parse_pool_id(s.pool_id, &grp, &member)) return arena_->peer_ptr(grp, member) != nullptr;
  {
    std::lock_guard<std::mutex> lk(mu_);
    if (pools_.count(s.pool_id)) return true;
  }
  const_cast<GpuFabric*>(this)->refresh_pools();  // a worker that joined after this fabric was created
  std::lock_guard<std::mutex> lk(mu_);
  return pools_.count(s.pool_id) > 0;
}

bool GpuFabric::is_local(const ShardPlacement& s) const {
  if (s.storage_class != StorageClass::RAM_GPU) return false;
  size_t grp = 0;
  int member = 0;
  if (arena_ && NvlsArena::parse_pool_id(s.pool_id, &grp, &member)) return member == arena_->rank();
  std::lock_guard<std::mutex> lk(mu_);
  auto it = pools_.find(s.pool_id);
  return it != pools_.end() && it->second.device == device_ && !it->second.ipc_opened;
}

GpuFabric::Path GpuFabric::classify(const ShardPlacement& s) const {
  if (s.storage_class != StorageClass::RAM_GPU) return PATH_PCIE;
  return is_local(s) ? PATH_HBM : PATH_NVLINK;
}

std::string GpuFabric::metrics_text() const {
  static const char* kPath[kNumPaths] = {"hbm", "nvlink", "pcie", "nvlink_multicast"};
  std::string out = "# HELP bb_fabric_bytes_total payload bytes moved by the fused transfer kernels\n# TYPE bb_fabric_bytes_total counter\n";
  const std::string g = std::to_string(device_);
  for (int d = 0; d < 2; ++d)
    for (int p = 0; p < kNumPaths; ++p) {
      if (d == 1 && p == PATH_MULTICAST) continue;
      out += "bb_fabric_bytes_total{gpu=\"" + g + "\",dir=\"" + (d == 0 ? "put" : "get") + "\",path=\"" + kPath[p] + "\"} " +
             std::to_string(bytes_[d][p].load(std::memory_order_relaxed)) + "\n";
    }
  out += "# TYPE bb_fabric_launches_total counter\nbb_fabric_launches_total{gpu=\"" + g + "\"} " + std::to_string(engine_->launches()) + "\n";
  out += "# TYPE bb_fabric_mapped_pools gauge\nbb_fabric_mapped_pools{gpu=\"" + g + "\",kind=\"all\"} " + std::to_string(mapped_pools()) + "\n";
  out += "bb_fabric_mapped_pools{gpu=\"" + g + "\",kind=\"dram\"} " + std::to_string(mapped_host_pools()) + "\n";
  out += "# TYPE bb_fabric_remaps_total counter\nbb_fabric_remaps_total{gpu=\"" + g + "\"} " + std::to_string(remaps_.load()) + "\n";
  return out;
}

Result<void*> GpuFabric::resolve(const ShardPlacement& s) {
  drop_if_stale(s);
  if (const auto* h = std::get_if<MemoryLocation>(&s.location)) {  // shared / pinned DRAM pool
    if (!ensure_host_pool(s.pool_id)) return ErrorCode::MEMORY_POOL_NOT_FOUND;
    std::lock_guard<std::mutex> lk(mu_);
    const Mapping& m = pools_.at(s.pool_id);
    if (h->remote_addr < m.remote_base || h->remote_addr - m.remote_base + s.length > m.size) return ErrorCode::MEMORY_ACCESS_ERROR;
    return static_cast<void*>(m.base + (h->remote_addr - m.remote_base));
  }
  const auto* g = std::get_if<GpuSlabLocation>(&s.location);
  if (!g) return ErrorCode::INVALID_ADDRESS;
  size_t grp = 0;
  int member = 0;
  if (arena_ && NvlsArena::parse_pool_id(s.pool_id, &grp, &member)) {
    auto* base = static_cast<uint8_t*>(arena_->peer_ptr(grp, member));
    if (!base) return ErrorCode::MEMORY_POOL_NOT_FOUND;
    if (g->offset + s.length > arena_->arena_bytes()) return ErrorCode::MEMORY_ACCESS_ERROR;
    return static_cast<void*>(base + g->offset);
  }
  for (int attempt = 0; attempt < 2; ++attempt) {
    {
      std::lock_guard<std::mutex> lk(mu_);
      auto it = pools_.find(s.pool_id);
      if (it != pools_.end()) {
        if (g->offset + s.length > it->second.size) return ErrorCode::MEMORY_ACCESS_ERROR;
        return static_cast<void*>(it->second.base + g->offset);
      }
    }
    if (attempt == 0) refresh_pools();  // a worker joined after we started
  }
  return ErrorCode::MEMORY_POOL_NOT_FOUND;
}

ErrorCode GpuFabric::copy_h2d(void* dev, const void* host, size_t n, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!cuda_ok(cudaSetDevice(device_), "cudaSetDevice") || !cuda_ok(cudaMemcpyAsync(dev, host, n, cudaMemcpyHostToDevice, st), "H2D") ||
      !cuda_ok(cudaStreamSynchronize(st), "sync"))
    return ErrorCode::FABRIC_ERROR;
  return ErrorCode::OK;
}

ErrorCode GpuFabric::copy_d2h(void* host, const void* dev, size_t n, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!cuda_ok(cudaSetDevice(device_), "cudaSetDevice") || !cuda_ok(cudaMemcpyAsync(host, dev, n, cudaMemcpyDeviceToHost, st), "D2H") ||
      !cuda_ok(cudaStreamSynchronize(st), "sync"))
    return ErrorCode::FABRIC_ERROR;
  return ErrorCode::OK;
}

// Segmented object: the item moves the slice of the object's segment list that this shard covers (the first and last
// segment trimmed by the engine), as the gather source (put) or the scatter destination (get).
static ErrorCode attach_segments(const client::DeviceShardOp& op, uint32_t flag, XferItem* it) {
  size_t first = 0, last = 0;
  uint64_t skip = 0, unused = 0;
  if (it->nbytes == 0) return ErrorCode::OK;
  if (!client::segment_slice(op.segs, op.nsegs, op.obj_offset, &first, &skip) ||
      !client::segment_slice(op.segs, op.nsegs, op.obj_offset + it->nbytes - 1, &last, &unused))
    return ErrorCode::INVALID_ARGUMENT;
  it->flags |= flag;
  it->segs = op.segs + first;
  it->nsegs = static_cast<uint32_t>(last - first + 1);
  it->seg_skip = skip;
  return ErrorCode::OK;
}

ErrorCode GpuFabric::build_put_items(const std::vector<client::DeviceShardOp>& ops, const std::vector<const void*>& dev_ptrs,
                                     std::vector<XferItem>* items, std::vector<size_t>* op_of_item) {
  items->reserve(ops.size());
  for (size_t k = 0; k < ops.size(); ++k) {
    const auto& op = ops[k];
    XferItem it;
    it.nbytes = op.placement->length;
    if (op.segs) {
      BB_TRY(attach_segments(op, XFER_GATHER, &it));
    } else {
      it.src = static_cast<const uint8_t*>(dev_ptrs[op.item]) + op.obj_offset;
    }
    // NVLS: the replica set is one whole multicast group at one offset -> a single multimem.st stream
    if (arena_ && !op.replicas.empty() && (it.nbytes & 15) == 0) {
      size_t grp = 0, g2 = 0;
      int m0 = 0, m2 = 0;
      const auto* loc0 = std::get_if<GpuSlabLocation>(&op.placement->location);
      bool mc_ok = loc0 && NvlsArena::parse_pool_id(op.placement->pool_id, &grp, &m0) && grp < arena_->num_groups() &&
                   arena_->member_of(grp) && arena_->mc_ptr(grp) && op.replicas.size() + 1 == arena_->members(grp).size();
      for (size_t r = 0; mc_ok && r < op.replicas.size(); ++r) {
        const auto* lr = std::get_if<GpuSlabLocation>(&op.replicas[r]->location);
        mc_ok = lr && lr->offset == loc0->offset && NvlsArena::parse_pool_id(op.replicas[r]->pool_id, &g2, &m2) && g2 == grp;
      }
      if (mc_ok) {
        it.dst[0] = static_cast<uint8_t*>(arena_->mc_ptr(grp)) + loc0->offset;
        it.ndst = 1;
        it.flags |= XFER_MULTIMEM;
        items->push_back(it);
        op_of_item->push_back(k);
        ++multicast_puts_;
        count(true, PATH_MULTICAST, it.nbytes);  // one egress stream, the switch replicates
        continue;
      }
    }
    auto d0 = resolve(*op.placement);
    if (!d0.ok()) return d0.error();
    it.dst[0] = d0.value();
    it.ndst = 1;
    count(true, classify(*op.placement), it.nbytes);
    for (const ShardPlacement* rp : op.replicas) count(true, classify(*rp), it.nbytes);
    size_t r = 0;
    for (; r < op.replicas.size() && it.ndst < kMaxDst; ++r) {
      auto d = resolve(*op.replicas[r]);
      if (!d.ok()) return d.error();
      it.dst[it.ndst++] = d.value();
    }
    items->push_back(it);
    op_of_item->push_back(k);
    // more replicas than one tile pass can fan out to: extra passes
    while (r < op.replicas.size()) {
      XferItem more;
      more.src = it.src;
      more.nbytes = it.nbytes;
      more.flags = it.flags & XFER_GATHER;
      more.segs = it.segs, more.nsegs = it.nsegs, more.seg_skip = it.seg_skip;
      more.ndst = 0;
      for (; r < op.replicas.size() && more.ndst < kMaxDst; ++r) {
        auto d = resolve(*op.replicas[r]);
        if (!d.ok()) return d.error();
        more.dst[more.ndst++] = d.value();
      }
      items->push_back(more);
      op_of_item->push_back(k);
    }
  }
  return ErrorCode::OK;
}

Result<uint64_t> GpuFabric::submit_put(const std::vector<client::DeviceShardOp>& ops, const std::vector<const void*>& dev_ptrs,
                                       ChecksumAlgo algo, void* stream) {
  BB_TRACE_SPAN("fabric.submit_put");
  std::vector<XferItem> items;
  InFlight fl;
  fl.nops = ops.size();
  ErrorCode ec = build_put_items(ops, dev_ptrs, &items, &fl.op_of_item);
  if (ec != ErrorCode::OK) return ec;
  auto t = engine_->submit(items, algo, stream);
  if (!t.ok()) return t.error();
  std::lock_guard<std::mutex> lk(mu_);
  inflight_[t.value()] = std::move(fl);
  return t.value();
}

ErrorCode GpuFabric::wait_put(uint64_t ticket, std::vector<uint64_t>* digests) {
  BB_TRACE_SPAN("fabric.wait_put");
  InFlight fl;
  {
    std::lock_guard<std::mutex> lk(mu_);
    auto it = inflight_.find(ticket);
    if (it == inflight_.end()) return ErrorCode::NOT_FOUND;
    fl = std::move(it->second);
    inflight_.erase(it);
  }
  XferResult res;
  ErrorCode ec = engine_->wait(ticket, &res);
  if (ec != ErrorCode::OK) return ec;
  last_ms_ = res.device_ms;
  total_ms_ += res.device_ms;
  if (digests) {
    digests->assign(fl.nops, 0);
    for (size_t i = fl.op_of_item.size(); i-- > 0;) (*digests)[fl.op_of_item[i]] = res.digest[i];
  }
  return ErrorCode::OK;
}

ErrorCode GpuFabric::put_fp8(const std::vector<client::DeviceFp8Op>& ops, void* stream, std::vector<uint64_t>* digests) {
  BB_TRACE_SPAN("fabric.put_fp8", ops.size());
  std::vector<Fp8Item> items;
  items.reserve(ops.size());
  for (const auto& op : ops) {
    auto d = resolve(*op.placement);
    if (!d.ok()) return d.error();
    Fp8Item it;
    it.wide = op.wide;
    it.packed = d.value();
    it.n_elems = op.n_elems;
    if (op.replicas.size() + 1 > kMaxDst) return ErrorCode::INVALID_ARGUMENT;
    for (const ShardPlacement* rp : op.replicas) {
      auto dr = resolve(*rp);
      if (!dr.ok()) return dr.error();
      it.more_packed[it.nreplicas - 1] = dr.value();
      ++it.nreplicas;
    }
    items.push_back(it);
  }
  XferResult res;
  ErrorCode ec = engine_->run_fp8(items, false, stream, &res);
  if (ec != ErrorCode::OK) return ec;
  last_ms_ = res.device_ms;
  total_ms_ += res.device_ms;
  if (digests) *digests = std::move(res.digest);
  return ErrorCode::OK;
}

ErrorCode GpuFabric::get_fp8(const std::vector<client::DeviceFp8Op>& ops, void* stream, std::vector<uint32_t>* status) {
  BB_TRACE_SPAN("fabric.get_fp8", ops.size());
  std::vector<Fp8Item> items;
  items.reserve(ops.size());
  for (const auto& op : ops) {
    auto d = resolve(*op.placement);
    if (!d.ok()) return d.error();
    Fp8Item it;
    it.wide = op.wide;
    it.packed = d.value();
    it.n_elems = op.n_elems;
    it.expect = op.placement->checksum;
    it.verify = true;
    items.push_back(it);
  }
  XferResult res;
  ErrorCode ec = engine_->run_fp8(items, true, stream, &res);
  if (ec != ErrorCode::OK) return ec;
  last_ms_ = res.device_ms;
  total_ms_ += res.device_ms;
  if (status) *status = std::move(res.status);
  return ErrorCode::OK;
}

ErrorCode GpuFabric::put_shards(const std::vector<client::DeviceShardOp>& ops, const std::vector<const void*>& dev_ptrs, ChecksumAlgo algo,
                                void* stream, std::vector<uint64_t>* digests) {
  auto t = submit_put(ops, dev_ptrs, algo, stream);
  if (!t.ok()) return t.error();
  return wait_put(t.value(), digests);
}

Result<uint64_t> GpuFabric::submit_get(const std::vector<client::DeviceShardOp>& ops, const std::vector<void*>& dev_ptrs, void* stream) {
  BB_TRACE_SPAN("fabric.submit_get");
  bool uniform = true;
  for (const auto& op : ops) uniform &= op.placement->checksum_algo == ops[0].placement->checksum_algo;
  InFlight fl;
  fl.nops = ops.size();
  if (!uniform || ops.empty()) {  // rare: objects written with different checksum algorithms in one batch
    fl.sync_done = true;
    ErrorCode ec = get_shards(ops, dev_ptrs, ChecksumAlgo::NONE, stream, &fl.sync_status);
    if (ec != ErrorCode::OK) return ec;
    std::lock_guard<std::mutex> lk(mu_);
    const uint64_t t = next_sync_ticket_++;
    inflight_[t] = std::move(fl);
    return t;
  }
  const ChecksumAlgo algo = ops[0].placement->checksum_algo;
  std::vector<XferItem> items;
  items.reserve(ops.size());
  for (const auto& op : ops) {
    XferItem it;
    auto s = resolve(*op.placement);
    if (!s.ok()) return s.error();
    it.src = s.value();
    it.ndst = 1;
    it.nbytes = op.placement->length;
    it.expect = op.placement->checksum;
    it.flags = algo == ChecksumAlgo::NONE ? 0u : static_cast<uint32_t>(XFER_VERIFY);
    if (op.segs) {
      BB_TRY(attach_segments(op, XFER_SCATTER, &it));
    } else {
      it.dst[0] = static_cast<uint8_t*>(dev_ptrs[op.item]) + op.obj_offset;
    }
    items.push_back(it);
    count(false, classify(*op.placement), it.nbytes);
  }
  auto t = engine_->submit(items, algo, stream);
  if (!t.ok()) return t.error();
  std::lock_guard<std::mutex> lk(mu_);
  inflight_[t.value()] = std::move(fl);
  return t.value();
}

ErrorCode GpuFabric::wait_get(uint64_t ticket, std::vector<uint32_t>* status) {
  BB_TRACE_SPAN("fabric.wait_get");
  InFlight fl;
  {
    std::lock_guard<std::mutex> lk(mu_);
    auto it = inflight_.find(ticket);
    if (it == inflight_.end()) return ErrorCode::NOT_FOUND;
    fl = std::move(it->second);
    inflight_.erase(it);
  }
  if (fl.sync_done) {
    if (status) *status = std::move(fl.sync_status);
    return ErrorCode::OK;
  }
  XferResult res;
  ErrorCode ec = engine_->wait(ticket, &res);
  if (ec != ErrorCode::OK) return ec;
  last_ms_ = res.device_ms;
  total_ms_ += res.device_ms;
  if (status) *status = std::move(res.status);
  return ErrorCode::OK;
}

ErrorCode GpuFabric::get_shards(const std::vector<client::DeviceShardOp>& ops, const std::vector<void*>& dev_ptrs, ChecksumAlgo,
                                void* stream, std::vector<uint32_t>* status) {
  if (status) status->assign(ops.size(), 0);
  // one launch per checksum algorithm present in the batch (normally exactly one)
  for (ChecksumAlgo algo : {ChecksumAlgo::XXH3, ChecksumAlgo::BBH64, ChecksumAlgo::CRC32C, ChecksumAlgo::NONE}) {
    std::vector<XferItem> items;
    std::vector<size_t> idx;
    for (size_t k = 0; k < ops.size(); ++k) {
      const auto& op = ops[k];
      if (op.placement->checksum_algo != algo) continue;
      XferItem it;
      auto s = resolve(*op.placement);
      if (!s.ok()) return s.error();
      it.src = s.value();
      it.ndst = 1;
      it.nbytes = op.placement->length;
      it.expect = op.placement->checksum;
      it.flags = algo == ChecksumAlgo::NONE ? 0u : static_cast<uint32_t>(XFER_VERIFY);
      if (op.segs) {
        BB_TRY(attach_segments(op, XFER_SCATTER, &it));
      } else {
        it.dst[0] = static_cast<uint8_t*>(dev_ptrs[op.item]) + op.obj_offset;
      }
      items.push_back(it);
      idx.push_back(k);
    }
    if (items.empty()) continue;
    XferResult res;
    ErrorCode ec = engine_->run(items, algo, stream, &res);
    if (ec != ErrorCode::OK) return ec;
    last_ms_ = res.device_ms;
  total_ms_ += res.device_ms;
    if (status)
      for (size_t i = 0; i < idx.size(); ++i) (*status)[idx[i]] = res.status[i];
  }
  return ErrorCode::OK;
}

}  // namespace bb::gpu
