// Python bindings of the control plane: types, allocator, coordination store, keystone, RPC,
// worker + storage backends, client SDK.  Result<T> maps to "value or raise BlackbirdError".
#include <pybind11/functional.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include "common/audit.h"
#include "common/tenant.h"
#include "alloc/allocator.h"
#include "client/blackbird_client.h"
#include "client/copy_mover.h"
#include "coord/etcd_coord.h"
#include "coord/coord.h"
#include "keystone/keystone_service.h"
#include "py/segments.h"
#include "rpc/rpc_service.h"
#include "rpc/wire.h"
#include "worker/worker_service.h"

namespace py = pybind11;
using namespace bb;

py::object bb_json_to_py(const Json& j);

namespace {

struct BlackbirdError : std::runtime_error {
  ErrorCode code;
  explicit BlackbirdError(ErrorCode c) : std::runtime_error(std::string(to_string(c))), code(c) {}
};

template <typename T>
T unwrap(Result<T> r) {
  if (!r.ok()) throw BlackbirdError(r.error());
  return std::move(r.value());
}

// Runs a native call that may block on the network with the GIL released (other Python threads -- e.g. an in-process
// proxy or server written in Python -- keep running); results are converted after the GIL is back.
template <typename F>
auto nogil(F&& f) {
  py::gil_scoped_release rel;
  return f();
}

// list[ErrorCode] for batch results.  pybind builds a fresh enum instance per element (~0.3 us); a batch of thousands of
// objects gets the cached instance of each code instead (enum members are immutable).  GIL held.
py::list ecs_to_py(const std::vector<ErrorCode>& v) {
  static std::unordered_map<int, PyObject*>* cache = new std::unordered_map<int, PyObject*>();  // lives as long as the interpreter
  py::list out(v.size());
  for (size_t i = 0; i < v.size(); ++i) {
    const int code = static_cast<int>(v[i]);
    auto it = cache->find(code);
    if (it == cache->end()) it = cache->emplace(code, py::cast(v[i]).release().ptr()).first;
    Py_INCREF(it->second);
    PyList_SET_ITEM(out.ptr(), static_cast<Py_ssize_t>(i), it->second);
  }
  return out;
}

py::dict scrub_to_py(const keystone::ScrubReport& r) {
  py::dict d;
  d["objects"] = r.objects;
  d["copies"] = r.copies;
  d["corrupt"] = r.corrupt;
  d["healed"] = r.healed;
  d["unrecoverable"] = r.unrecoverable;
  d["unreachable"] = r.unreachable;
  return d;
}

py::list tenant_usage_to_py(const std::vector<keystone::TenantUsage>& v) {
  py::list out;
  for (const auto& u : v) {
    py::dict d;
    d["name"] = u.name;
    d["used_bytes"] = u.used_bytes;
    d["objects"] = u.objects;
    d["quota_bytes"] = u.quota_bytes;
    d["max_objects"] = u.max_objects;
    out.append(d);
  }
  return out;
}

// RAII TenantScope as a Python context manager: in-process callers act on behalf of a tenant (ACL + budget apply).
struct PyTenantScope {
  std::string name;
  std::unique_ptr<TenantScope> scope;
};

py::object location_to_py(const LocationDetail& l) {
  py::dict d;
  if (auto* m = std::get_if<MemoryLocation>(&l)) {
    d["kind"] = "memory";
    d["remote_addr"] = m->remote_addr;
    d["rkey"] = m->rkey;
    d["size"] = m->size;
  } else if (auto* f = std::get_if<FileLocation>(&l)) {
    d["kind"] = "file";
    d["file_path"] = f->file_path;
    d["file_offset"] = f->file_offset;
  } else if (auto* c = std::get_if<CxlMemoryLocation>(&l)) {
    d["kind"] = "cxl";
    d["device_id"] = c->device_id;
    d["region_id"] = c->region_id;
    d["offset"] = c->offset;
    d["size"] = c->size;
  } else if (auto* g = std::get_if<GpuSlabLocation>(&l)) {
    d["kind"] = "gpu";
    d["device_rank"] = g->device_rank;
    d["slab_id"] = g->slab_id;
    d["offset"] = g->offset;
    d["size"] = g->size;
  }
  return d;
}

// Python callables captured by C++ callbacks may be released on arbitrary native threads:
// the deleter takes the GIL before dropping the reference.
template <typename T>
std::shared_ptr<T> gil_safe_holder(T obj) {
  return std::shared_ptr<T>(new T(std::move(obj)), [](T* p) {
    if (Py_IsInitialized()) {
      py::gil_scoped_acquire g;
      delete p;
    } else {
      p->release();  // interpreter is gone: leak the reference instead of touching it
      delete p;
    }
  });
}

// py results of batch calls: list of (ErrorCode, value-or-None)
template <typename T, typename F>
py::list results_to_py(const std::vector<Result<T>>& v, F&& conv) {
  py::list out;
  for (const auto& r : v) out.append(py::make_tuple(r.error(), r.ok() ? py::object(conv(r.value())) : py::object(py::none())));
  return out;
}

}  // namespace

void bind_control(py::module_& m) {
  static py::exception<BlackbirdError> exc(m, "BlackbirdError");
  py::register_exception_translator([](std::exception_ptr p) {
    try {
      if (p) std::rethrow_exception(p);
    } catch (const BlackbirdError& e) {
      // attach the code to the exception instance
      PyObject* inst = PyObject_CallFunction(exc.ptr(), "s", e.what());
      if (inst) {
        py::object code = py::cast(e.code);
        PyObject_SetAttrString(inst, "code", code.ptr());
        PyErr_SetObject(exc.ptr(), inst);
        Py_DECREF(inst);
      }
    }
  });

  // ---------------------------------------------------------------- types
  py::enum_<StorageClass>(m, "StorageClass")
      .value("STORAGE_UNSPECIFIED", StorageClass::STORAGE_UNSPECIFIED)
      .value("RAM_CPU", StorageClass::RAM_CPU)
      .value("RAM_GPU", StorageClass::RAM_GPU)
      .value("NVME", StorageClass::NVME)
      .value("SSD", StorageClass::SSD)
      .value("HDD", StorageClass::HDD)
      .value("CXL_MEMORY", StorageClass::CXL_MEMORY)
      .value("CXL_TYPE2_DEVICE", StorageClass::CXL_TYPE2_DEVICE)
      .value("CUSTOM", StorageClass::CUSTOM);
  m.def("parse_storage_class", [](const std::string& s) -> py::object {
    auto c = parse_storage_class(s);
    return c ? py::cast(*c) : py::none();
  });
  m.def("tier_rank", &tier_rank);

  py::class_<TransportEndpoint>(m, "TransportEndpoint")
      .def(py::init<>())
      .def_readwrite("ip", &TransportEndpoint::ip)
      .def_readwrite("port", &TransportEndpoint::port)
      .def_property("worker_key", [](const TransportEndpoint& e) { return py::bytes(reinterpret_cast<const char*>(e.worker_key.data()), e.worker_key.size()); },
                    [](TransportEndpoint& e, const std::string& b) { e.worker_key.assign(b.begin(), b.end()); });

  py::class_<ShardPlacement>(m, "ShardPlacement")
      .def(py::init<>())
      .def_readwrite("pool_id", &ShardPlacement::pool_id)
      .def_readwrite("worker_id", &ShardPlacement::worker_id)
      .def_readwrite("endpoint", &ShardPlacement::endpoint)
      .def_readwrite("storage_class", &ShardPlacement::storage_class)
      .def_readwrite("length", &ShardPlacement::length)
      .def_readwrite("checksum", &ShardPlacement::checksum)
      .def_readwrite("checksum_algo", &ShardPlacement::checksum_algo)
      .def_property_readonly("location", [](const ShardPlacement& s) { return location_to_py(s.location); })
      .def_property_readonly("offset", [](const ShardPlacement& s) -> uint64_t {
        if (auto* g = std::get_if<GpuSlabLocation>(&s.location)) return g->offset;
        if (auto* f = std::get_if<FileLocation>(&s.location)) return f->file_offset;
        if (auto* c = std::get_if<CxlMemoryLocation>(&s.location)) return c->offset;
        if (auto* mm = std::get_if<MemoryLocation>(&s.location)) return mm->remote_addr;
        return 0;
      });

  py::class_<CopyPlacement>(m, "CopyPlacement")
      .def(py::init<>())
      .def_readwrite("copy_index", &CopyPlacement::copy_index)
      .def_readwrite("shards", &CopyPlacement::shards)
      .def("shards_size", &CopyPlacement::shards_size);

  py::class_<WorkerConfig>(m, "WorkerConfig")
      .def(py::init([](size_t replication_factor, size_t max_workers_per_copy, bool enable_soft_pin, std::string preferred_node,
                       std::vector<StorageClass> preferred_classes, uint64_t ttl_ms, bool enable_locality_awareness,
                       bool prefer_contiguous, size_t min_shard_size, ChecksumAlgo checksum, bool pack_fp8, bool symmetric_replicas) {
             WorkerConfig c;
             c.replication_factor = replication_factor;
             c.max_workers_per_copy = max_workers_per_copy;
             c.enable_soft_pin = enable_soft_pin;
             c.preferred_node = std::move(preferred_node);
             c.preferred_classes = std::move(preferred_classes);
             c.ttl_ms = ttl_ms;
             c.enable_locality_awareness = enable_locality_awareness;
             c.prefer_contiguous = prefer_contiguous;
             c.min_shard_size = min_shard_size;
             c.checksum = checksum;
             c.pack_fp8 = pack_fp8;
             c.symmetric_replicas = symmetric_replicas;
             return c;
           }),
           py::arg("replication_factor") = DEFAULT_REPLICATION_FACTOR, py::arg("max_workers_per_copy") = DEFAULT_MAX_WORKERS_PER_COPY,
           py::arg("enable_soft_pin") = false, py::arg("preferred_node") = "", py::arg("preferred_classes") = std::vector<StorageClass>{},
           py::arg("ttl_ms") = 30ull * 60 * 1000, py::arg("enable_locality_awareness") = true, py::arg("prefer_contiguous") = false,
           py::arg("min_shard_size") = 4096, py::arg("checksum") = ChecksumAlgo::BBH64, py::arg("pack_fp8") = false,
           py::arg("symmetric_replicas") = false)
      .def_readwrite("replication_factor", &WorkerConfig::replication_factor)
      .def_readwrite("max_workers_per_copy", &WorkerConfig::max_workers_per_copy)
      .def_readwrite("enable_soft_pin", &WorkerConfig::enable_soft_pin)
      .def_readwrite("preferred_node", &WorkerConfig::preferred_node)
      .def_readwrite("preferred_classes", &WorkerConfig::preferred_classes)
      .def_readwrite("ttl_ms", &WorkerConfig::ttl_ms)
      .def_readwrite("enable_locality_awareness", &WorkerConfig::enable_locality_awareness)
      .def_readwrite("prefer_contiguous", &WorkerConfig::prefer_contiguous)
      .def_readwrite("min_shard_size", &WorkerConfig::min_shard_size)
      .def_readwrite("checksum", &WorkerConfig::checksum)
      .def_readwrite("pack_fp8", &WorkerConfig::pack_fp8)
      .def_readwrite("symmetric_replicas", &WorkerConfig::symmetric_replicas)
      .def("to_json", [](const WorkerConfig& c) { return to_json(c).dump(); });

  py::class_<ClusterStats>(m, "ClusterStats")
      .def_readonly("total_workers", &ClusterStats::total_workers)
      .def_readonly("total_memory_pools", &ClusterStats::total_memory_pools)
      .def_readonly("total_objects", &ClusterStats::total_objects)
      .def_readonly("total_capacity", &ClusterStats::total_capacity)
      .def_readonly("used_capacity", &ClusterStats::used_capacity)
      .def_readonly("avg_utilization", &ClusterStats::avg_utilization)
      .def_readonly("pending_objects", &ClusterStats::pending_objects)
      .def_readonly("active_clients", &ClusterStats::active_clients);

  py::class_<MemoryPool>(m, "MemoryPool")
      .def(py::init([](std::string id, uint64_t size, StorageClass sc, std::string node_id, std::string worker_id, std::string endpoint,
                       uint64_t remote_addr, std::string rkey_hex, int gpu_device_id, double max_bw_gbps, std::string fabric_domain,
                       std::string mount_path) {
             MemoryPool p;
             p.id = std::move(id);
             p.size = size;
             p.storage_class = sc;
             p.node_id = std::move(node_id);
             p.worker_id = std::move(worker_id);
             p.ucx_endpoint = std::move(endpoint);
             p.ucx_remote_addr = remote_addr;
             p.base_addr = remote_addr;
             p.ucx_rkey_hex = std::move(rkey_hex);
             p.gpu_device_id = gpu_device_id;
             p.max_bw_gbps = max_bw_gbps;
             p.fabric_domain = std::move(fabric_domain);
             p.mount_path = std::move(mount_path);
             return p;
           }),
           py::arg("id"), py::arg("size"), py::arg("storage_class") = StorageClass::RAM_CPU, py::arg("node_id") = "node-a",
           py::arg("worker_id") = "", py::arg("endpoint") = "127.0.0.1:12345", py::arg("remote_addr") = 0x1000000,
           py::arg("rkey_hex") = "deadbeef", py::arg("gpu_device_id") = -1, py::arg("max_bw_gbps") = 0.0,
           py::arg("fabric_domain") = "", py::arg("mount_path") = "")
      .def_readwrite("id", &MemoryPool::id)
      .def_readwrite("node_id", &MemoryPool::node_id)
      .def_readwrite("worker_id", &MemoryPool::worker_id)
      .def_readwrite("size", &MemoryPool::size)
      .def_readwrite("used", &MemoryPool::used)
      .def_readwrite("storage_class", &MemoryPool::storage_class)
      .def_readwrite("ucx_endpoint", &MemoryPool::ucx_endpoint)
      .def_readwrite("ucx_remote_addr", &MemoryPool::ucx_remote_addr)
      .def_readwrite("ucx_rkey_hex", &MemoryPool::ucx_rkey_hex)
      .def_readwrite("gpu_device_id", &MemoryPool::gpu_device_id)
      .def_readwrite("max_bw_gbps", &MemoryPool::max_bw_gbps)
      .def_readwrite("fabric_domain", &MemoryPool::fabric_domain)
      .def("available", &MemoryPool::available)
      .def("utilization", &MemoryPool::utilization)
      .def("to_json", [](const MemoryPool& p) { return to_json(p).dump(); })
      .def_static("from_json", [](const std::string& s) {
        auto j = Json::parse(s);
        if (!j) throw py::value_error("bad json");
        return unwrap(memory_pool_from_json(*j));
      });

  py::class_<KeystoneConfig>(m, "KeystoneConfig")
      .def(py::init<>())
      .def_static("from_yaml", &KeystoneConfig::from_yaml)
      .def_readwrite("cluster_id", &KeystoneConfig::cluster_id)
      .def_readwrite("etcd_endpoints", &KeystoneConfig::etcd_endpoints)
      .def_readwrite("listen_address", &KeystoneConfig::listen_address)
      .def_readwrite("http_metrics_port", &KeystoneConfig::http_metrics_port)
      .def_readwrite("service_id", &KeystoneConfig::service_id)
      .def_readwrite("enable_gc", &KeystoneConfig::enable_gc)
      .def_readwrite("enable_ha", &KeystoneConfig::enable_ha)
      .def_readwrite("eviction_ratio", &KeystoneConfig::eviction_ratio)
      .def_readwrite("high_watermark", &KeystoneConfig::high_watermark)
      .def_readwrite("client_ttl_sec", &KeystoneConfig::client_ttl_sec)
      .def_readwrite("worker_heartbeat_ttl_sec", &KeystoneConfig::worker_heartbeat_ttl_sec)
      .def_readwrite("service_registration_ttl_sec", &KeystoneConfig::service_registration_ttl_sec)
      .def_readwrite("service_refresh_interval_sec", &KeystoneConfig::service_refresh_interval_sec)
      .def_readwrite("gc_interval_sec", &KeystoneConfig::gc_interval_sec)
      .def_readwrite("scrub_objects_per_round", &KeystoneConfig::scrub_objects_per_round)
      .def_readwrite("tenants_file", &KeystoneConfig::tenants_file)
      .def_readwrite("health_check_interval_sec", &KeystoneConfig::health_check_interval_sec)
      .def_readwrite("max_replicas", &KeystoneConfig::max_replicas)
      .def_readwrite("default_replicas", &KeystoneConfig::default_replicas)
      .def_readwrite("rpc_threads", &KeystoneConfig::rpc_threads)
      .def_readwrite("rpc_busy_poll_us", &KeystoneConfig::rpc_busy_poll_us)
      .def_readwrite("tier_policy", &KeystoneConfig::tier_policy)
      .def_readwrite("promote_after_reads", &KeystoneConfig::promote_after_reads)
      .def_readwrite("compaction_fragmentation_threshold", &KeystoneConfig::compaction_fragmentation_threshold)
      .def_readwrite("wal_path", &KeystoneConfig::wal_path)
      .def_readwrite("wal_fsync", &KeystoneConfig::wal_fsync)
      .def_readwrite("enable_reservations", &KeystoneConfig::enable_reservations)
      .def_readwrite("reservation_ttl_ms", &KeystoneConfig::reservation_ttl_ms)
      .def_readwrite("wal_snapshot_mb", &KeystoneConfig::wal_snapshot_mb)
      .def_readwrite("log_level", &KeystoneConfig::log_level)
      .def("validate", [](const KeystoneConfig& c) {
        std::string err;
        ErrorCode ec = c.validate(&err);
        return py::make_tuple(ec, err);
      });

  m.def("bytes_to_hex", [](const std::string& b) { return bytes_to_hex(std::vector<uint8_t>(b.begin(), b.end())); });
  m.def("hex_to_bytes", [](const std::string& h) -> py::object {
    auto b = hex_to_bytes(h);
    if (!b) return py::none();
    return py::bytes(reinterpret_cast<const char*>(b->data()), b->size());
  });

  // ---------------------------------------------------------------- allocator
  using alloc::AllocationRequest;
  using alloc::AllocationResult;
  using alloc::PoolAllocator;
  using alloc::Range;
  using alloc::RangeAllocator;
  py::class_<Range>(m, "Range")
      .def(py::init<uint64_t, uint64_t>())
      .def_readwrite("offset", &Range::offset)
      .def_readwrite("length", &Range::length)
      .def("end", &Range::end)
      .def("adjacent_to", &Range::adjacent_to)
      .def("merge_with", &Range::merge_with);
  py::class_<PoolAllocator>(m, "PoolAllocator")
      .def(py::init<const MemoryPool&, uint64_t>(), py::arg("pool"), py::arg("align") = PoolAllocator::kDefaultAlign)
      .def("allocate", [](PoolAllocator& a, uint64_t size, bool best) -> py::object {
        std::optional<Range> r;
        {
          py::gil_scoped_release rel;
          r = a.allocate(size, best);
        }
        return r ? py::cast(*r) : py::none();
      }, py::arg("size"), py::arg("prefer_best_fit") = true)
      .def("allocate_at", &PoolAllocator::allocate_at)
      .def("free", &PoolAllocator::free, py::call_guard<py::gil_scoped_release>())
      .def("total_free", &PoolAllocator::total_free)
      .def("largest_free_block", &PoolAllocator::largest_free_block)
      .def("fragmentation_ratio", &PoolAllocator::fragmentation_ratio)
      .def("can_allocate", &PoolAllocator::can_allocate)
      .def("free_ranges", &PoolAllocator::free_ranges)
      .def("pool_id", &PoolAllocator::pool_id);
  py::class_<AllocationRequest>(m, "AllocationRequest")
      .def(py::init([](std::string key, size_t data_size, size_t replication_factor, size_t max_workers_per_copy,
                       std::vector<StorageClass> preferred_classes, std::string preferred_node, bool enable_locality_awareness,
                       bool enable_striping, bool prefer_contiguous, size_t min_shard_size, bool strict_min_shard,
                       bool symmetric_replicas, std::string client_node) {
             AllocationRequest r;
             r.object_key = std::move(key);
             r.data_size = data_size;
             r.replication_factor = replication_factor;
             r.max_workers_per_copy = max_workers_per_copy;
             r.preferred_classes = std::move(preferred_classes);
             r.preferred_node = std::move(preferred_node);
             r.enable_locality_awareness = enable_locality_awareness;
             r.enable_striping = enable_striping;
             r.prefer_contiguous = prefer_contiguous;
             r.min_shard_size = min_shard_size;
             r.strict_min_shard = strict_min_shard;
             r.symmetric_replicas = symmetric_replicas;
             r.client_node = std::move(client_node);
             return r;
           }),
           py::arg("object_key"), py::arg("data_size"), py::arg("replication_factor") = 1, py::arg("max_workers_per_copy") = 1,
           py::arg("preferred_classes") = std::vector<StorageClass>{}, py::arg("preferred_node") = "",
           py::arg("enable_locality_awareness") = true, py::arg("enable_striping") = true, py::arg("prefer_contiguous") = false,
           py::arg("min_shard_size") = 4096, py::arg("strict_min_shard") = false, py::arg("symmetric_replicas") = false,
           py::arg("client_node") = "");
  py::class_<AllocationResult>(m, "AllocationResult")
      .def_readonly("copies", &AllocationResult::copies)
      .def_readonly("total_shards_created", &AllocationResult::total_shards_created)
      .def_readonly("pools_used", &AllocationResult::pools_used)
      .def_property_readonly("required_spillover", [](const AllocationResult& r) { return r.stats.required_spillover; })
      .def_property_readonly("avg_shard_size", [](const AllocationResult& r) { return r.stats.avg_shard_size; });
  py::class_<alloc::AllocatorStats>(m, "AllocatorStats")
      .def_readonly("total_allocated_bytes", &alloc::AllocatorStats::total_allocated_bytes)
      .def_readonly("total_free_bytes", &alloc::AllocatorStats::total_free_bytes)
      .def_readonly("total_objects", &alloc::AllocatorStats::total_objects)
      .def_readonly("total_shards", &alloc::AllocatorStats::total_shards)
      .def_readonly("fragmentation_ratio", &alloc::AllocatorStats::fragmentation_ratio);
  py::class_<RangeAllocator>(m, "RangeAllocator")
      .def(py::init<>())
      .def("allocate", [](RangeAllocator& a, const AllocationRequest& r, const std::unordered_map<MemoryPoolId, MemoryPool>& pools) {
        return unwrap(a.allocate(r, pools));
      })
      .def("free", &RangeAllocator::free)
      .def("get_stats", [](RangeAllocator& a, py::object sc) {
        return a.get_stats(sc.is_none() ? std::nullopt : std::optional<StorageClass>(sc.cast<StorageClass>()));
      }, py::arg("storage_class") = py::none())
      .def("get_free_space", &RangeAllocator::get_free_space)
      .def("can_allocate", &RangeAllocator::can_allocate)
      .def("pool_used_bytes", &RangeAllocator::pool_used_bytes)
      .def("forget_pool", &RangeAllocator::forget_pool);

  // ---------------------------------------------------------------- coordination
  using coord::CoordService;
  using coord::CoordStore;
  using coord::MemCoord;
  // Every call may block on the network (RemoteCoord, EtcdCoord): the GIL is released around the C++ call, which also
  // lets an in-process Python server (tests/fake_etcd.py) answer it.
  py::class_<CoordStore, std::shared_ptr<CoordStore>>(m, "CoordStore")
      .def("put", &CoordStore::put, py::arg("key"), py::arg("value"), py::arg("lease") = 0, py::call_guard<py::gil_scoped_release>())
      .def("get", [](CoordStore& s, const std::string& k) -> py::object {
        Result<std::string> r = ErrorCode::INTERNAL_ERROR;
        {
          py::gil_scoped_release rel;
          r = s.get(k);
        }
        if (!r.ok()) return py::none();
        return py::bytes(r.value());
      })
      .def("delete", &CoordStore::del, py::call_guard<py::gil_scoped_release>())
      .def("get_with_prefix", [](CoordStore& s, const std::string& p) {
        Result<std::vector<coord::KeyValue>> r = ErrorCode::INTERNAL_ERROR;
        {
          py::gil_scoped_release rel;
          r = s.get_with_prefix(p);
        }
        py::list out;
        for (auto& kv : unwrap(std::move(r))) out.append(py::make_tuple(kv.key, py::bytes(kv.value), kv.mod_revision, kv.lease));
        return out;
      })
      .def("del_prefix", [](CoordStore& s, const std::string& p) { return unwrap(s.del_prefix(p)); }, py::call_guard<py::gil_scoped_release>())
      .def("grant_lease", [](CoordStore& s, int64_t ttl) { return unwrap(s.grant_lease(ttl)); }, py::call_guard<py::gil_scoped_release>())
      .def("keep_alive", &CoordStore::keep_alive, py::call_guard<py::gil_scoped_release>())
      .def("revoke_lease", &CoordStore::revoke_lease, py::call_guard<py::gil_scoped_release>())
      .def("lease_remaining_ms", [](CoordStore& s, LeaseId l) { return unwrap(s.lease_remaining_ms(l)); }, py::call_guard<py::gil_scoped_release>())
      .def("put_if_absent", [](CoordStore& s, const std::string& k, const std::string& v, LeaseId l) { return unwrap(s.put_if_absent(k, v, l)); },
           py::arg("key"), py::arg("value"), py::arg("lease") = 0, py::call_guard<py::gil_scoped_release>())
      .def("compare_and_swap", [](CoordStore& s, const std::string& k, const std::string& e, const std::string& v, LeaseId l) {
        return unwrap(s.compare_and_swap(k, e, v, l));
      }, py::arg("key"), py::arg("expected"), py::arg("value"), py::arg("lease") = 0, py::call_guard<py::gil_scoped_release>())
      .def("compare_and_delete", [](CoordStore& s, const std::string& k, const std::string& e) { return unwrap(s.compare_and_delete(k, e)); },
           py::call_guard<py::gil_scoped_release>())
      .def("guarded_put", [](CoordStore& s, const std::string& g, int64_t rev, const std::string& k, const std::string& v) {
        return unwrap(s.guarded_put(g, rev, k, v));
      }, py::arg("guard_key"), py::arg("guard_create_revision"), py::arg("key"), py::arg("value"), py::call_guard<py::gil_scoped_release>())
      .def("guarded_del", [](CoordStore& s, const std::string& g, int64_t rev, const std::string& k) { return unwrap(s.guarded_del(g, rev, k)); },
           py::call_guard<py::gil_scoped_release>())
      .def("get_kv", [](CoordStore& s, const std::string& k) -> py::object {
        Result<coord::KeyValue> r = ErrorCode::INTERNAL_ERROR;
        {
          py::gil_scoped_release rel;
          r = s.get_kv(k);
        }
        if (!r.ok()) return py::none();
        py::dict d;
        d["key"] = r.value().key;
        d["value"] = py::bytes(r.value().value);
        d["create_revision"] = r.value().create_revision;
        d["mod_revision"] = r.value().mod_revision;
        d["lease"] = r.value().lease;
        return d;
      })
      .def("watch_prefix", [](CoordStore& s, const std::string& prefix, py::function cb) {
        auto holder = gil_safe_holder(std::move(cb));
        return unwrap(s.watch_prefix(prefix, [holder](const coord::WatchEvent& ev) {
          py::gil_scoped_acquire g;
          try {
            (*holder)(ev.type == coord::EventType::DELETE ? "DELETE" : "PUT", ev.key, py::bytes(ev.value), ev.revision);
          } catch (py::error_already_set& e) {
            e.discard_as_unraisable("watch callback");
          }
        }));
      }, py::call_guard<py::gil_scoped_release>())
      .def("unwatch", &CoordStore::unwatch, py::call_guard<py::gil_scoped_release>())
      .def("revision", &CoordStore::revision, py::call_guard<py::gil_scoped_release>());
  py::class_<MemCoord, CoordStore, std::shared_ptr<MemCoord>>(m, "MemCoord")
      // The destructor joins the dispatch thread, which may be waiting for the GIL to deliver an event to a Python
      // watch callback: release the GIL while the store is torn down.
      .def(py::init([] {
        return std::shared_ptr<MemCoord>(new MemCoord(), [](MemCoord* p) {
          py::gil_scoped_release rel;
          delete p;
        });
      }))
      .def("advance_time_ms", &MemCoord::advance_time_ms, py::call_guard<py::gil_scoped_release>())
      .def("flush_events", &MemCoord::flush_events, py::call_guard<py::gil_scoped_release>())
      .def("lease_count", &MemCoord::lease_count)
      .def("key_count", &MemCoord::key_count)
      .def("open_durable", &MemCoord::open_durable, py::arg("dir"), py::arg("fsync") = true, py::arg("snapshot_bytes") = 64ull << 20,
           py::call_guard<py::gil_scoped_release>(), "Persist every mutation under `dir` (log + snapshots); replays what is there.")
      .def_property_readonly("durable", &MemCoord::durable)
      .def_property_readonly("recovered_records", &MemCoord::recovered_records);
  py::class_<coord::RemoteCoord, CoordStore, std::shared_ptr<coord::RemoteCoord>>(m, "RemoteCoord")
      .def(py::init<>())
      .def("connect", &coord::RemoteCoord::connect, py::arg("endpoints"), py::arg("timeout_ms") = 3000)
      .def("close", &coord::RemoteCoord::close, py::call_guard<py::gil_scoped_release>())
      .def_property_readonly("reconnects", &coord::RemoteCoord::reconnects);
  py::class_<coord::EtcdCoord, CoordStore, std::shared_ptr<coord::EtcdCoord>>(m, "EtcdCoord")
      .def(py::init<>())
      .def("connect", &coord::EtcdCoord::connect, py::arg("endpoints"), py::arg("timeout_ms") = 3000, py::call_guard<py::gil_scoped_release>())
      .def("close", &coord::EtcdCoord::close, py::call_guard<py::gil_scoped_release>())
      .def_property_readonly("requests", &coord::EtcdCoord::requests);
  py::class_<coord::CoordServer>(m, "CoordServer")
      .def(py::init([](std::shared_ptr<MemCoord> st) { return std::make_unique<coord::CoordServer>(std::move(st)); }), py::arg("store") = nullptr)
      .def("start", &coord::CoordServer::start, py::arg("host") = "127.0.0.1", py::arg("port") = 0)
      .def("stop", &coord::CoordServer::stop, py::call_guard<py::gil_scoped_release>())
      .def_property_readonly("port", &coord::CoordServer::port)
      .def("store", &coord::CoordServer::store);
  m.def("shared_mem_coord", &coord::shared_mem_coord);
  m.def("drop_shared_mem_coord", &coord::drop_shared_mem_coord);

  py::class_<CoordService, std::shared_ptr<CoordService>>(m, "CoordService")
      .def(py::init<const std::string&>(), py::arg("endpoints") = "")
      .def(py::init<std::shared_ptr<CoordStore>>())
      .def("connect", &CoordService::connect)
      .def("is_connected", &CoordService::is_connected)
      .def("store", &CoordService::store)
      .def("put", &CoordService::put)
      .def("get", [](CoordService& s, const std::string& k) -> py::object {
        std::string v;
        return s.get(k, v) == ErrorCode::OK ? py::object(py::bytes(v)) : py::object(py::none());
      })
      .def("delete", &CoordService::del)
      .def("put_with_ttl", &CoordService::put_with_ttl)
      .def("register_service", &CoordService::register_service)
      .def("discover_service", [](CoordService& s, const std::string& name) {
        std::vector<std::string> a;
        s.discover_service(name, a);
        return a;
      })
      .def("unregister_service", &CoordService::unregister_service)
      .def("campaign_leader", [](CoordService& s, const std::string& e, const std::string& c, int64_t ttl) {
        bool won = false;
        ErrorCode ec = s.campaign_leader(e, c, ttl, won);
        return py::make_tuple(ec, won);
      })
      .def("get_leader", [](CoordService& s, const std::string& e) -> py::object {
        std::string l;
        return s.get_leader(e, l) == ErrorCode::OK ? py::object(py::str(l)) : py::object(py::none());
      })
      .def("resign_leader", &CoordService::resign_leader)
      .def("refresh_leadership", &CoordService::refresh_leadership, py::call_guard<py::gil_scoped_release>())
      .def("leader_term", &CoordService::leader_term)
      .def("fenced_put", &CoordService::fenced_put, py::call_guard<py::gil_scoped_release>())
      .def("fenced_del", &CoordService::fenced_del, py::call_guard<py::gil_scoped_release>());

  // ---------------------------------------------------------------- keystone
  using keystone::KeystoneService;
  using keystone::PutStartItem;
  py::enum_<keystone::ObjectState>(m, "ObjectState").value("PENDING", keystone::ObjectState::PENDING).value("COMPLETE", keystone::ObjectState::COMPLETE);
  py::class_<KeystoneService, std::shared_ptr<KeystoneService>>(m, "KeystoneService")
      .def(py::init<const KeystoneConfig&, std::shared_ptr<CoordService>>(), py::arg("config"), py::arg("coord") = nullptr)
      .def("initialize", &KeystoneService::initialize, py::call_guard<py::gil_scoped_release>())
      .def("start", &KeystoneService::start, py::call_guard<py::gil_scoped_release>())
      .def("stop", &KeystoneService::stop, py::call_guard<py::gil_scoped_release>())
      .def("is_running", &KeystoneService::is_running)
      .def("is_leader", &KeystoneService::is_leader)
      .def("leader_term", &KeystoneService::leader_term)
      .def("object_exists", [](KeystoneService& k, const std::string& key) { return unwrap(k.object_exists(key)); })
      .def("get_workers", [](KeystoneService& k, const std::string& key) { return unwrap(k.get_workers(key)); })
      .def("put_start", [](KeystoneService& k, const std::string& key, size_t size, const WorkerConfig& c, const std::string& client,
                           const std::string& node) { return unwrap(k.put_start(key, size, c, client, node)); },
           py::arg("key"), py::arg("size"), py::arg("config") = WorkerConfig{}, py::arg("client_id") = "", py::arg("client_node") = "")
      .def("put_complete", [](KeystoneService& k, const std::string& key, const keystone::ShardChecksums& s) { return k.put_complete(key, s); },
           py::arg("key"), py::arg("checksums") = keystone::ShardChecksums{})
      .def("put_cancel", &KeystoneService::put_cancel)
      .def("remove_object", &KeystoneService::remove_object)
      .def("migrate_object", &KeystoneService::migrate_object, py::call_guard<py::gil_scoped_release>())
      .def("run_promotion_once", &KeystoneService::run_promotion_once, py::call_guard<py::gil_scoped_release>())
      .def("remove_all_objects", [](KeystoneService& k) { return unwrap(k.remove_all_objects()); })
      .def("batch_object_exists", [](KeystoneService& k, const std::vector<std::string>& keys) {
        return results_to_py(k.batch_object_exists(keys), [](bool b) { return py::bool_(b); });
      })
      .def("batch_get_workers", [](KeystoneService& k, const std::vector<std::string>& keys) {
        return results_to_py(k.batch_get_workers(keys), [](const std::vector<CopyPlacement>& v) { return py::cast(v); });
      })
      .def("batch_put_start", [](KeystoneService& k, const std::vector<std::string>& keys, const std::vector<size_t>& sizes, const WorkerConfig& c) {
        std::vector<PutStartItem> items;
        for (size_t i = 0; i < keys.size(); ++i) items.push_back({keys[i], i < sizes.size() ? sizes[i] : 0, c});
        return results_to_py(k.batch_put_start(items), [](const std::vector<CopyPlacement>& v) { return py::cast(v); });
      })
      .def("batch_put_complete", [](KeystoneService& k, const std::vector<std::string>& keys) { return k.batch_put_complete(keys); })
      .def("batch_put_cancel", &KeystoneService::batch_put_cancel)
      .def("batch_remove_object", &KeystoneService::batch_remove_object)
      .def("get_cluster_stats", [](KeystoneService& k) { return unwrap(k.get_cluster_stats()); })
      .def("get_view_version", &KeystoneService::get_view_version)
      .def("get_memory_pools", [](KeystoneService& k) {
        std::vector<MemoryPool> v;
        k.get_memory_pools(v);
        return v;
      })
      .def("get_workers_info", [](KeystoneService& k) {
        std::vector<keystone::WorkerInfo> v;
        k.get_workers_info(v);
        py::list out;
        for (const auto& w : v) {
          py::dict d;
          d["worker_id"] = w.worker_id;
          d["node_id"] = w.node_id;
          d["endpoint"] = w.endpoint;
          d["pools"] = w.pools;
          out.append(d);
        }
        return out;
      })
      .def("remove_worker", &KeystoneService::remove_worker, py::call_guard<py::gil_scoped_release>())
      .def("drain_worker", [](KeystoneService& k, const std::string& id) { return unwrap(nogil([&] { return k.drain_worker(id); })); },
           "move every object off the worker (old copies keep serving), then remove it; returns the number of objects moved")
      .def("run_compaction_once", &KeystoneService::run_compaction_once, py::call_guard<py::gil_scoped_release>())
      .def("compact_pool", [](KeystoneService& k, const std::string& pool, size_t max_moves) { return unwrap(k.compact_pool(pool, max_moves)); },
           py::arg("pool"), py::arg("max_moves") = 64, py::call_guard<py::gil_scoped_release>())
      .def("register_memory_pool", &KeystoneService::register_memory_pool)
      .def("register_worker", [](KeystoneService& k, const std::string& id, const std::string& node, const std::string& ep) {
        WorkerRecord r;
        r.worker_id = id;
        r.node_id = node;
        r.rpc_endpoint = ep;
        return k.register_worker(r);
      }, py::arg("worker_id"), py::arg("node_id") = "", py::arg("endpoint") = "")
      .def("worker_heartbeat", &KeystoneService::worker_heartbeat)
      .def("handle_worker_death", &KeystoneService::handle_worker_death, py::call_guard<py::gil_scoped_release>())
      .def("client_register", [](KeystoneService& k, const std::string& n) { return unwrap(k.client_register(n)); })
      .def("client_ping", [](KeystoneService& k, const std::string& id) { return unwrap(k.client_ping(id)); })
      .def("run_gc_once", &KeystoneService::run_gc_once, py::call_guard<py::gil_scoped_release>())
      .def("run_eviction_once", &KeystoneService::run_eviction_once, py::call_guard<py::gil_scoped_release>())
      .def("run_repair_once", &KeystoneService::run_repair_once, py::call_guard<py::gil_scoped_release>())
      .def("tier_utilization", &KeystoneService::tier_utilization)
      .def("metrics_text", &KeystoneService::metrics_text)
      .def("stats_json", [](KeystoneService& k) { return bb_json_to_py(k.stats_json()); })
      .def("allocator_stats", &KeystoneService::allocator_stats)
      .def("object_info", [](KeystoneService& k, const std::string& key) {
        auto o = unwrap(k.get_object_info(key));
        py::dict d;
        d["size"] = o.size;
        d["state"] = o.state;
        d["copies"] = o.copies;
        d["soft_pin"] = o.config.enable_soft_pin;
        d["ttl_ms"] = o.config.ttl_ms;
        return d;
      })
      .def("install_reservation_hooks", [](KeystoneService& k) { k.set_reservation_hooks(client::make_data_server_reservation_hooks()); },
           "Reservation protocol over the workers' data servers (takes effect with KeystoneConfig.enable_reservations).")
      .def("tenant_usage", [](KeystoneService& k) { return tenant_usage_to_py(k.tenant_usage()); },
           "per tenant: used_bytes (size x replicas of its live objects), objects, quota_bytes, max_objects")
      .def("scrub", [](KeystoneService& k, const std::string& prefix, size_t max_objects) { return scrub_to_py(unwrap(nogil([&] { return k.scrub(prefix, max_objects); }))); },
           py::arg("prefix") = "", py::arg("max_objects") = 0)
      .def("install_data_server_verifier", [](KeystoneService& k) { k.set_copy_verifier(client::make_data_server_verifier()); })
      .def("install_data_server_mover", [](KeystoneService& k) { k.set_copy_verifier(client::make_data_server_verifier()); k.set_copy_mover(client::make_data_server_mover()); },
           "Tier demotion / re-replication move bytes through the workers' data servers (the default in bb-keystone).")
      // Python-implemented copy mover (tests): fn(key, src_copy, dst_copy, algo) -> (ErrorCode, [shard checksums])
      .def("set_copy_mover", [](KeystoneService& k, py::object fn) {
        if (fn.is_none()) {
          k.set_copy_mover(nullptr);
          return;
        }
        auto holder = gil_safe_holder(std::move(fn));
        k.set_copy_mover([holder](const ObjectKey& key, const CopyPlacement& src, CopyPlacement& dst, ChecksumAlgo algo) {
          py::gil_scoped_acquire g;
          try {
            py::tuple r = (*holder)(key, src, dst, algo);
            ErrorCode ec = r[0].cast<ErrorCode>();
            if (ec == ErrorCode::OK && r.size() > 1) {
              auto sums = r[1].cast<std::vector<uint64_t>>();
              for (size_t i = 0; i < sums.size() && i < dst.shards.size(); ++i) dst.shards[i].checksum = sums[i];
            }
            return ec;
          } catch (py::error_already_set& e) {
            e.discard_as_unraisable("copy mover");
            return ErrorCode::INTERNAL_ERROR;
          }
        });
      });

  py::class_<rpc::RpcService>(m, "RpcService")
      .def(py::init<std::shared_ptr<KeystoneService>, const KeystoneConfig&>())
      .def("start", &rpc::RpcService::start, py::call_guard<py::gil_scoped_release>())
      .def("stop", &rpc::RpcService::stop, py::call_guard<py::gil_scoped_release>())
      .def_property_readonly("rpc_port", &rpc::RpcService::rpc_port)
      .def_property_readonly("http_port", &rpc::RpcService::http_port)
      .def_property_readonly("requests_served", &rpc::RpcService::requests_served)
      .def_property_readonly("shm_requests_served", &rpc::RpcService::shm_requests_served)
      .def_property_readonly("shm_channels", &rpc::RpcService::shm_channels);

  py::class_<rpc::KeystoneApi, std::shared_ptr<rpc::KeystoneApi>>(m, "KeystoneApi")
      .def("object_exists", [](rpc::KeystoneApi& k, const std::string& key) { return unwrap(k.object_exists(key)); }, py::call_guard<py::gil_scoped_release>())
      .def("get_workers", [](rpc::KeystoneApi& k, const std::string& key) { return unwrap(k.get_workers(key)); }, py::call_guard<py::gil_scoped_release>())
      .def("put_start", [](rpc::KeystoneApi& k, const std::string& key, size_t size, const WorkerConfig& c) { return unwrap(nogil([&] { return k.put_start(key, size, c); })); },
           py::arg("key"), py::arg("size"), py::arg("config") = WorkerConfig{})
      .def("put_complete", [](rpc::KeystoneApi& k, const std::string& key, const keystone::ShardChecksums& s) { return k.put_complete(key, s); },
           py::arg("key"), py::arg("checksums") = keystone::ShardChecksums{}, py::call_guard<py::gil_scoped_release>())
      .def("put_cancel", &rpc::KeystoneApi::put_cancel, py::call_guard<py::gil_scoped_release>())
      .def("remove_object", &rpc::KeystoneApi::remove_object, py::call_guard<py::gil_scoped_release>())
      .def("migrate_object", &rpc::KeystoneApi::migrate_object, py::call_guard<py::gil_scoped_release>())
      .def("remove_all_objects", [](rpc::KeystoneApi& k) { return unwrap(k.remove_all_objects()); }, py::call_guard<py::gil_scoped_release>())
      .def("get_cluster_stats", [](rpc::KeystoneApi& k) { return unwrap(k.get_cluster_stats()); }, py::call_guard<py::gil_scoped_release>())
      .def("get_view_version", [](rpc::KeystoneApi& k) { return unwrap(k.get_view_version()); }, py::call_guard<py::gil_scoped_release>())
      .def("batch_object_exists", [](rpc::KeystoneApi& k, const std::vector<std::string>& keys) {
        return results_to_py(nogil([&] { return k.batch_object_exists(keys); }), [](bool b) { return py::bool_(b); });
      })
      .def("batch_get_workers", [](rpc::KeystoneApi& k, const std::vector<std::string>& keys) {
        return results_to_py(nogil([&] { return k.batch_get_workers(keys); }), [](const std::vector<CopyPlacement>& v) { return py::cast(v); });
      })
      .def("batch_put_start", [](rpc::KeystoneApi& k, const std::vector<std::string>& keys, const std::vector<size_t>& sizes, const WorkerConfig& c) {
        std::vector<PutStartItem> items;
        for (size_t i = 0; i < keys.size(); ++i) items.push_back({keys[i], i < sizes.size() ? sizes[i] : 0, c});
        return results_to_py(nogil([&] { return k.batch_put_start(items); }), [](const std::vector<CopyPlacement>& v) { return py::cast(v); });
      })
      // (network calls: never with the GIL held -- an in-process Python peer, e.g. a test's fake server, could not answer)
      .def("batch_put_complete", [](rpc::KeystoneApi& k, const std::vector<std::string>& keys) { return ecs_to_py(nogil([&] { return k.batch_put_complete(keys, {}); })); })
      .def("batch_put_cancel", [](rpc::KeystoneApi& k, const std::vector<std::string>& keys) { return ecs_to_py(nogil([&] { return k.batch_put_cancel(keys); })); })
      .def("batch_remove_object", [](rpc::KeystoneApi& k, const std::vector<std::string>& keys) { return ecs_to_py(nogil([&] { return k.batch_remove_object(keys); })); })
      .def("get_memory_pools", [](rpc::KeystoneApi& k) { return unwrap(nogil([&] { return k.get_memory_pools(); })); })
      .def("get_workers_info", [](rpc::KeystoneApi& k) {
        py::list out;
        for (const auto& w : unwrap(nogil([&] { return k.get_workers_info(); }))) {
          py::dict d;
          d["worker_id"] = w.worker_id;
          d["node_id"] = w.node_id;
          d["endpoint"] = w.endpoint;
          d["heartbeat_age_ms"] = w.heartbeat_age_ms;
          d["pools"] = w.pools;
          out.append(d);
        }
        return out;
      })
      .def("remove_worker", &rpc::KeystoneApi::remove_worker, py::call_guard<py::gil_scoped_release>())
      .def("drain_worker", [](rpc::KeystoneApi& k, const std::string& id) { return unwrap(nogil([&] { return k.drain_worker(id); })); })
      .def("tenant_usage", [](rpc::KeystoneApi& k) { return tenant_usage_to_py(unwrap(nogil([&] { return k.tenant_usage(); }))); },
           "what each tenant holds against its budget (a tenant connection sees only its own line)")
      .def("scrub", [](rpc::KeystoneApi& k, const std::string& prefix, size_t max_objects) { return scrub_to_py(unwrap(nogil([&] { return k.scrub(prefix, max_objects); }))); },
           py::arg("prefix") = "", py::arg("max_objects") = 0)
      .def("compact_pool", [](rpc::KeystoneApi& k, const std::string& pool, size_t max_moves) { return unwrap(nogil([&] { return k.compact_pool(pool, max_moves); })); },
           py::arg("pool"), py::arg("max_moves") = 64)
      .def("list_objects", [](rpc::KeystoneApi& k, const std::string& prefix, size_t limit, const std::string& after) {
        py::list out;
        for (const auto& o : unwrap(nogil([&] { return k.list_objects(prefix, limit, after); }))) out.append(py::make_tuple(o.key, o.size, o.copies, o.tier));
        return out;
      }, py::arg("prefix") = "", py::arg("limit") = 0, py::arg("start_after") = "", "[(key, size, copies, tier)] in key order")
      .def("client_register", [](rpc::KeystoneApi& k, const std::string& n) { return unwrap(nogil([&] { return k.client_register(n); })); })
      .def("client_ping", [](rpc::KeystoneApi& k, const std::string& id) { return unwrap(nogil([&] { return k.client_ping(id); })); })
      .def("register_memory_pool", &rpc::KeystoneApi::register_memory_pool, py::call_guard<py::gil_scoped_release>())
      .def("worker_heartbeat", &rpc::KeystoneApi::worker_heartbeat, py::call_guard<py::gil_scoped_release>());
  py::class_<rpc::KeystoneRpcClient, rpc::KeystoneApi, std::shared_ptr<rpc::KeystoneRpcClient>>(m, "KeystoneRpcClient")
      .def(py::init<>())
      .def("connect", [](rpc::KeystoneRpcClient& c, const std::string& host, uint16_t port, int timeout_ms) { return c.connect(host, port, timeout_ms); },
           py::arg("host"), py::arg("port"), py::arg("timeout_ms") = 3000, py::call_guard<py::gil_scoped_release>())
      .def("connect_any", [](rpc::KeystoneRpcClient& c, const std::vector<std::string>& eps, int timeout_ms) { return c.connect_any(eps, timeout_ms); },
           py::arg("endpoints"), py::arg("timeout_ms") = 3000, py::call_guard<py::gil_scoped_release>())
      .def("set_timeout_ms", &rpc::KeystoneRpcClient::set_timeout_ms)
      .def("set_failover_budget_ms", &rpc::KeystoneRpcClient::set_failover_budget_ms)
      .def("active_endpoint", &rpc::KeystoneRpcClient::active_endpoint)
      .def("failovers", &rpc::KeystoneRpcClient::failovers)
      .def("connected", &rpc::KeystoneRpcClient::connected);
  py::class_<rpc::LocalKeystoneApi, rpc::KeystoneApi, std::shared_ptr<rpc::LocalKeystoneApi>>(m, "LocalKeystoneApi")
      .def(py::init<std::shared_ptr<KeystoneService>>());

  m.def("http_get", [](const std::string& host, uint16_t port, const std::string& path) {
    int status = 0;
    Result<std::string> r = ErrorCode::INTERNAL_ERROR;
    {
      py::gil_scoped_release rel;
      r = net::http_get(host, port, path, &status);
    }
    if (!r.ok()) throw BlackbirdError(r.error());
    return py::make_tuple(status, r.value());
  });

  // ---------------------------------------------------------------- worker + backends
  using worker::StorageBackend;
  py::class_<worker::ReservationToken>(m, "ReservationToken")
      .def_readonly("token_id", &worker::ReservationToken::token_id)
      .def_readonly("pool_id", &worker::ReservationToken::pool_id)
      .def_readonly("remote_addr", &worker::ReservationToken::remote_addr)
      .def_readonly("rkey", &worker::ReservationToken::rkey)
      .def_readonly("size", &worker::ReservationToken::size);
  py::class_<worker::StorageStats>(m, "StorageStats")
      .def_readonly("total_capacity", &worker::StorageStats::total_capacity)
      .def_readonly("used_capacity", &worker::StorageStats::used_capacity)
      .def_readonly("available_capacity", &worker::StorageStats::available_capacity)
      .def_readonly("num_reservations", &worker::StorageStats::num_reservations)
      .def_readonly("num_committed_shards", &worker::StorageStats::num_committed_shards)
      .def_readonly("utilization", &worker::StorageStats::utilization)
      .def_readonly("bytes_written", &worker::StorageStats::bytes_written)
      .def_readonly("bytes_read", &worker::StorageStats::bytes_read)
      .def_readonly("io_errors", &worker::StorageStats::io_errors);
  py::class_<StorageBackend>(m, "StorageBackend")
      .def("get_storage_class", &StorageBackend::get_storage_class)
      .def("get_total_capacity", &StorageBackend::get_total_capacity)
      .def("get_used_capacity", &StorageBackend::get_used_capacity)
      .def("get_available_capacity", &StorageBackend::get_available_capacity)
      .def("get_base_address", &StorageBackend::get_base_address)
      .def("get_rkey", &StorageBackend::get_rkey)
      .def("registration_key_hex", &StorageBackend::registration_key_hex)
      .def("initialize", &StorageBackend::initialize, py::call_guard<py::gil_scoped_release>())
      .def("shutdown", &StorageBackend::shutdown, py::call_guard<py::gil_scoped_release>())
      .def("reserve_shard", [](StorageBackend& b, uint64_t size, const std::string& hint) { return unwrap(b.reserve_shard(size, hint)); },
           py::arg("size"), py::arg("hint") = "", py::call_guard<py::gil_scoped_release>())
      .def("commit_shard", &StorageBackend::commit_shard, py::call_guard<py::gil_scoped_release>())
      .def("abort_shard", &StorageBackend::abort_shard)
      .def("free_shard", &StorageBackend::free_shard)
      .def("get_stats", &StorageBackend::get_stats)
      .def("write", [](StorageBackend& b, uint64_t off, py::buffer data) {
        py::buffer_info i = data.request();
        py::gil_scoped_release rel;
        return b.write(off, i.ptr, static_cast<uint64_t>(i.size * i.itemsize));
      })
      .def("read", [](StorageBackend& b, uint64_t off, uint64_t len) {
        std::string out(len, '\0');
        ErrorCode ec;
        {
          py::gil_scoped_release rel;
          ec = b.read(off, out.data(), len);
        }
        if (ec != ErrorCode::OK) throw BlackbirdError(ec);
        return py::bytes(out);
      })
      .def("flush", &StorageBackend::flush)
      .def("cuda_accessible", &StorageBackend::cuda_accessible)
      .def_property_readonly("device_copies", &StorageBackend::device_copies, "tier moves done by the fused kernel")
      .def("set_pool_id", &StorageBackend::set_pool_id)
      .def("set_reservation_ttl_ms", &StorageBackend::set_reservation_ttl_ms)
      .def("has_direct_ptr", [](StorageBackend& b) { return b.direct_ptr(0) != nullptr; });
  py::class_<worker::IoUringDiskBackend, StorageBackend>(m, "IoUringDiskBackend")
      .def_property_readonly("sqes_submitted", &worker::IoUringDiskBackend::sqes_submitted)
      .def_property_readonly("fixed_sqes", &worker::IoUringDiskBackend::fixed_sqes)
      .def_property_readonly("using_uring", &worker::IoUringDiskBackend::using_uring)
      .def_property_readonly("using_direct_io", &worker::IoUringDiskBackend::using_direct_io)
      .def_property_readonly("file_path", &worker::IoUringDiskBackend::file_path)
      .def("recovered_extents", [](worker::IoUringDiskBackend& b) {
        py::list out;
        for (const auto& e : b.recovered_extents()) out.append(py::make_tuple(e.offset, e.size, e.crc));
        return out;
      });
  py::class_<worker::CxlMemoryBackend, StorageBackend>(m, "CxlMemoryBackend")
      .def_property_readonly("is_dax", &worker::CxlMemoryBackend::is_dax)
      .def_property_readonly("numa_bound", &worker::CxlMemoryBackend::numa_bound)
      .def("region_id", &worker::CxlMemoryBackend::region_id);
  py::class_<worker::MmapDiskBackend, StorageBackend>(m, "MmapDiskBackend").def_property_readonly("file_path", &worker::MmapDiskBackend::file_path);
  py::class_<worker::RamBackend, StorageBackend>(m, "RamBackend")
      .def_property_readonly("shared_path", &worker::RamBackend::shared_path)
      .def_property_readonly("pinned", &worker::RamBackend::pinned);
  m.def("create_storage_backend", [](StorageClass sc, uint64_t capacity, const std::string& mount_path, uint32_t queue_depth, int numa_node,
                                      const std::string& pool_id, bool shared_memory, const std::string& at_rest_key) -> std::unique_ptr<StorageBackend> {
    worker::BackendOptions o;
    o.mount_path = mount_path;
    o.queue_depth = queue_depth;
    o.numa_node = numa_node;
    o.shared_memory = shared_memory;
    o.at_rest_key = at_rest_key;
    o.at_rest_scope = pool_id;
    auto b = worker::create_storage_backend(sc, capacity, o);
    if (b && !pool_id.empty()) b->set_pool_id(pool_id);
    return b;
  }, py::arg("storage_class"), py::arg("capacity"), py::arg("mount_path") = "", py::arg("queue_depth") = 64, py::arg("numa_node") = -1,
     py::arg("pool_id") = "", py::arg("shared_memory") = false, py::arg("at_rest_key") = "");
  // Maps another worker's shared RAM pool (registration key = hex of "file:<path>") and returns its first `n` bytes
  // starting at `offset` (test / diagnostics helper for the mapping the GPU fabric performs).
  m.def("read_shared_pool", [](const std::string& key_hex, uint64_t pool_size, uint64_t offset, uint64_t n) -> py::object {
    auto raw = hex_to_bytes(key_hex);
    if (!raw || offset + n > pool_size) return py::none();
    void* p = worker::map_shared_pool(*raw, pool_size);
    if (!p) return py::none();
    py::bytes out(static_cast<const char*>(p) + offset, n);
    worker::unmap_shared_pool(p, pool_size);
    return out;
  });
  m.def("io_uring_supported", &worker::IoUring::supported);
  m.def("attach_loopback_transport", [](std::shared_ptr<client::BlackbirdClient> c, std::shared_ptr<client::BlackbirdClient> io, bool reach_disk_tiers) {
    c->set_device_transport(std::make_shared<client::HostLoopbackTransport>(std::move(io), reach_disk_tiers));
  }, py::arg("client"), py::arg("io_client"), py::arg("reach_disk_tiers") = false,
        "CPU stand-in for the GPU fabric: the device batch API of `client` moves host buffers through `io_client`'s host data paths");
  m.def("set_cluster_token", &net::set_cluster_token, "shared-secret gate of the RPC servers / clients of this process (net/tcp.h)");
  m.def("set_cluster_token_ro", &net::set_cluster_token_ro, "second secret: members that prove only this one are read-only (net/tcp.h)");
  // tenants (common/tenant.h): named principals with their own secret, key-prefix grants and a budget
  m.def("set_tenants", [](const std::vector<py::dict>& rows) {
    std::vector<Tenant> v;
    for (const auto& d : rows) {
      Tenant t;
      t.name = py::cast<std::string>(d["name"]);
      t.secret = py::cast<std::string>(d["secret"]);
      if (d.contains("read")) t.read_prefixes = py::cast<std::vector<std::string>>(d["read"]);
      if (d.contains("write")) t.write_prefixes = py::cast<std::vector<std::string>>(d["write"]);
      if (d.contains("quota_bytes")) t.quota_bytes = py::cast<uint64_t>(d["quota_bytes"]);
      if (d.contains("max_objects")) t.max_objects = py::cast<uint64_t>(d["max_objects"]);
      if (d.contains("admin")) t.admin = py::cast<bool>(d["admin"]);
      if (t.name.empty() || t.name.size() > kMaxTenantName || t.secret.empty()) throw py::value_error("tenant needs a name (1..64 bytes) and a secret");
      v.push_back(std::move(t));
    }
    set_tenants(std::move(v));
  }, "install the process-wide tenant table: [{name, secret, read: [...], write: [...], quota_bytes, max_objects, admin}]");
  m.def("load_tenants_file", [](const std::string& path) {
    std::string err;
    if (load_tenants_file(path, &err) != ErrorCode::OK) throw py::value_error(err);
  });
  m.def("load_tenants_text", [](const std::string& yaml) {
    std::string err;
    if (load_tenants_text(yaml, &err) != ErrorCode::OK) throw py::value_error(err);
  });
  m.def("reload_tenants_if_changed", &reload_tenants_if_changed);
  m.def("tenant_names", &tenant_names);
  m.def("set_client_tenant", &set_client_tenant, py::arg("name"), py::arg("secret"),
        "the identity RPC clients of this process present when they hold no member token (\"\", \"\" = none)");
  m.def("tenant_may", [](const std::string& name, const std::string& key, bool write) {
    auto t = find_tenant(name);
    return t && (write ? t->may_write(key) : t->may_read(key));
  }, py::arg("tenant"), py::arg("key"), py::arg("write") = false);
  py::class_<PyTenantScope>(m, "TenantScope", "with TenantScope(name): in-process Keystone calls of this thread run on behalf of that tenant")
      .def(py::init([](const std::string& name) {
        if (!find_tenant(name)) throw py::value_error("unknown tenant " + name);
        return PyTenantScope{name, nullptr};
      }))
      .def("__enter__", [](PyTenantScope& s) -> PyTenantScope& {
        s.scope = std::make_unique<TenantScope>(find_tenant(s.name));
        return s;
      }, py::return_value_policy::reference)
      .def("__exit__", [](PyTenantScope& s, py::object, py::object, py::object) { s.scope.reset(); });
  m.def("audit_open", &audit::open, "append-only JSON-lines audit trail of this process's servers (common/audit.h); \"\" closes it");
  m.def("audit_events_written", &audit::events_written);
  m.def("set_http_token", &net::set_http_token, "bearer token of the HTTP endpoints (/metrics, /stats) served and fetched by this process; \"\" = open");
  m.def("set_transport_encryption", &net::set_transport_encryption, "secure mode of the RPC protocol: AES-256-GCM on every frame, keyed from the cluster token");
  m.def("transport_encryption", &net::transport_encryption);
  // test hook: AES-256-CTR by byte offset (net::OffsetCipher) over a buffer
  m.def("offset_cipher_crypt", [](const py::bytes& key32, const py::bytes& nonce8, uint64_t offset, const py::bytes& data) -> py::object {
    const std::string k = key32, n = nonce8, d = data;
    if (k.size() != net::kAeadKey || n.size() != 8) throw py::value_error("key = 32 bytes, nonce = 8 bytes");
    net::OffsetCipher c;
    if (!c.set_key(reinterpret_cast<const uint8_t*>(k.data()), reinterpret_cast<const uint8_t*>(n.data()))) return py::none();
    std::string out(d.size(), '\0');
    if (!c.crypt(offset, d.data(), out.data(), d.size())) return py::none();
    return py::bytes(out);
  });
  m.def("aead_available", [] {
    std::string why;
    const bool ok = net::Aead::available(&why);
    return py::make_tuple(ok, why);
  });
  m.def("cluster_token", &net::cluster_token);

  // CXL transport / pool configuration (reference include/blackbird/transport/cxl_transport_config.h)
  py::enum_<CxlInterconnectType>(m, "CxlInterconnectType")
      .value("CXL_MEM", CxlInterconnectType::CXL_MEM)
      .value("CXL_CACHE", CxlInterconnectType::CXL_CACHE)
      .value("CXL_IO", CxlInterconnectType::CXL_IO)
      .value("CXL_FABRIC", CxlInterconnectType::CXL_FABRIC)
      .value("HYBRID", CxlInterconnectType::HYBRID);
  py::enum_<CxlTransportProtocol>(m, "CxlTransportProtocol")
      .value("DIRECT_CXL", CxlTransportProtocol::DIRECT_CXL)
      .value("RDMA_OVER_CXL", CxlTransportProtocol::RDMA_OVER_CXL)
      .value("NVLINK", CxlTransportProtocol::NVLINK)
      .value("CUSTOM", CxlTransportProtocol::CUSTOM);
  m.def("cxl_interconnect_name", [](CxlInterconnectType t) { return std::string(to_string(t)); });
  m.def("cxl_protocol_name", [](CxlTransportProtocol t) { return std::string(to_string(t)); });
  py::class_<CxlTransportConfig>(m, "CxlTransportConfig")
      .def(py::init<>())
      .def_readwrite("interconnect_type", &CxlTransportConfig::interconnect_type)
      .def_readwrite("transport_protocol", &CxlTransportConfig::transport_protocol)
      .def_readwrite("enable_fabric_manager", &CxlTransportConfig::enable_fabric_manager)
      .def_readwrite("fabric_manager_endpoint", &CxlTransportConfig::fabric_manager_endpoint)
      .def_readwrite("max_transfer_size", &CxlTransportConfig::max_transfer_size)
      .def_readwrite("queue_depth", &CxlTransportConfig::queue_depth)
      .def_readwrite("enable_zero_copy", &CxlTransportConfig::enable_zero_copy)
      .def_readwrite("enable_multipath", &CxlTransportConfig::enable_multipath)
      .def_readwrite("fallback_transports", &CxlTransportConfig::fallback_transports)
      .def_readwrite("priority", &CxlTransportConfig::priority)
      .def_readwrite("bandwidth_limit_gbps", &CxlTransportConfig::bandwidth_limit_gbps)
      .def_readwrite("enable_cxl_hdm", &CxlTransportConfig::enable_cxl_hdm)
      .def_readwrite("enable_cxl_switch", &CxlTransportConfig::enable_cxl_switch)
      .def_readwrite("cxl_port_id", &CxlTransportConfig::cxl_port_id)
      .def("resolve_interconnects", &CxlTransportConfig::resolve_interconnects, py::arg("cxl_present"), py::arg("have_gpu"))
      .def("to_dict", [](const CxlTransportConfig& c) { return bb_json_to_py(c.to_json()); });
  py::class_<CxlMemoryPoolConfig>(m, "CxlMemoryPoolConfig")
      .def(py::init<>())
      .def_readwrite("device_id", &CxlMemoryPoolConfig::device_id)
      .def_readwrite("device_path", &CxlMemoryPoolConfig::device_path)
      .def_readwrite("dax_device", &CxlMemoryPoolConfig::dax_device)
      .def_readwrite("capacity", &CxlMemoryPoolConfig::capacity)
      .def_readwrite("latency_ns", &CxlMemoryPoolConfig::latency_ns)
      .def_readwrite("bandwidth_gbps", &CxlMemoryPoolConfig::bandwidth_gbps)
      .def_readwrite("is_persistent", &CxlMemoryPoolConfig::is_persistent)
      .def_readwrite("enable_numa_binding", &CxlMemoryPoolConfig::enable_numa_binding)
      .def_readwrite("numa_node", &CxlMemoryPoolConfig::numa_node)
      .def_readwrite("interleave_ways", &CxlMemoryPoolConfig::interleave_ways)
      .def_readwrite("interleave_granularity", &CxlMemoryPoolConfig::interleave_granularity)
      .def_readwrite("cache_line_size", &CxlMemoryPoolConfig::cache_line_size)
      .def("to_dict", [](const CxlMemoryPoolConfig& c) { return bb_json_to_py(c.to_json()); });
  py::class_<TierRule>(m, "TierRule")
      .def(py::init([](std::string sc, uint64_t lo, uint64_t hi) { return TierRule{std::move(sc), lo, hi}; }), py::arg("storage_class"),
           py::arg("min_size") = 0, py::arg("max_size") = UINT64_MAX)
      .def_readwrite("storage_class", &TierRule::storage_class)
      .def_readwrite("min_size", &TierRule::min_size)
      .def_readwrite("max_size", &TierRule::max_size);
  m.def("tier_classes_for_size", &tier_classes_for_size);
  py::class_<worker::StoragePoolConfig>(m, "StoragePoolConfig")
      .def(py::init([](std::string pool_id, StorageClass sc, uint64_t size, std::string mount_path, int gpu_device_id) {
             worker::StoragePoolConfig c;
             c.pool_id = std::move(pool_id);
             c.storage_class = sc;
             c.size_bytes = size;
             c.mount_path = std::move(mount_path);
             c.gpu_device_id = gpu_device_id;
             return c;
           }),
           py::arg("pool_id"), py::arg("storage_class"), py::arg("size_bytes"), py::arg("mount_path") = "", py::arg("gpu_device_id") = 0)
      .def_readwrite("pool_id", &worker::StoragePoolConfig::pool_id)
      .def_readwrite("storage_class", &worker::StoragePoolConfig::storage_class)
      .def_readwrite("size_bytes", &worker::StoragePoolConfig::size_bytes)
      .def_readwrite("mount_path", &worker::StoragePoolConfig::mount_path)
      .def_readwrite("gpu_device_id", &worker::StoragePoolConfig::gpu_device_id)
      .def_readwrite("numa_node", &worker::StoragePoolConfig::numa_node)
      .def_readwrite("pin_memory", &worker::StoragePoolConfig::pin_memory)
      .def_readwrite("shared_memory", &worker::StoragePoolConfig::shared_memory)
      .def_readwrite("encrypt_at_rest", &worker::StoragePoolConfig::encrypt_at_rest)
      .def_readwrite("cxl", &worker::StoragePoolConfig::cxl);
  py::class_<worker::WorkerServiceConfig>(m, "WorkerServiceConfig")
      .def(py::init<>())
      .def_static("from_yaml", &worker::load_worker_config_from_file)
      .def_readwrite("worker_id", &worker::WorkerServiceConfig::worker_id)
      .def_readwrite("http_metrics_port", &worker::WorkerServiceConfig::http_metrics_port)
      .def_readwrite("node_id", &worker::WorkerServiceConfig::node_id)
      .def_readwrite("cluster_id", &worker::WorkerServiceConfig::cluster_id)
      .def_readwrite("etcd_endpoints", &worker::WorkerServiceConfig::etcd_endpoints)
      .def_readwrite("keystone_address", &worker::WorkerServiceConfig::keystone_address)
      .def_readwrite("rpc_endpoint", &worker::WorkerServiceConfig::rpc_endpoint)
      .def_readwrite("ucx_endpoint", &worker::WorkerServiceConfig::ucx_endpoint)
      .def_readwrite("interconnects", &worker::WorkerServiceConfig::interconnects)
      .def_readwrite("max_bw_gbps", &worker::WorkerServiceConfig::max_bw_gbps)
      .def_readwrite("numa_node", &worker::WorkerServiceConfig::numa_node)
      .def_readwrite("lease_ttl_sec", &worker::WorkerServiceConfig::lease_ttl_sec)
      .def_readwrite("heartbeat_interval_sec", &worker::WorkerServiceConfig::heartbeat_interval_sec)
      .def_readwrite("allocation_poll_interval_ms", &worker::WorkerServiceConfig::allocation_poll_interval_ms)
      .def_readwrite("at_rest_key", &worker::WorkerServiceConfig::at_rest_key)
      .def_readwrite("fabric_domain", &worker::WorkerServiceConfig::fabric_domain)
      .def_readwrite("transport", &worker::WorkerServiceConfig::transport)
      .def_readwrite("has_transport", &worker::WorkerServiceConfig::has_transport)
      .def_readwrite("preferred_tiers", &worker::WorkerServiceConfig::preferred_tiers)
      .def_readwrite("storage_pools", &worker::WorkerServiceConfig::storage_pools);
  py::class_<worker::WorkerService, std::shared_ptr<worker::WorkerService>>(m, "WorkerService")
      .def(py::init<const worker::WorkerServiceConfig&, std::shared_ptr<CoordService>, std::shared_ptr<rpc::KeystoneApi>>(), py::arg("config"),
           py::arg("coord") = nullptr, py::arg("keystone") = nullptr)
      .def("create_storage_pools_from_config", &worker::WorkerService::create_storage_pools_from_config)
      .def("initialize", &worker::WorkerService::initialize, py::call_guard<py::gil_scoped_release>())
      .def("start", &worker::WorkerService::start, py::call_guard<py::gil_scoped_release>())
      .def("stop", &worker::WorkerService::stop, py::call_guard<py::gil_scoped_release>())
      .def("is_running", &worker::WorkerService::is_running)
      .def("get_stats", [](worker::WorkerService& w) { return bb_json_to_py(w.get_stats()); })
      .def("advertised_pools", &worker::WorkerService::advertised_pools)
      .def("data_endpoint", &worker::WorkerService::data_endpoint)
      .def("metrics_text", &worker::WorkerService::metrics_text)
      .def_property_readonly("http_port", &worker::WorkerService::http_port)
      .def("inject_fault", &worker::WorkerService::inject_fault)
      .def("reap_reservations", &worker::WorkerService::reap_reservations, py::call_guard<py::gil_scoped_release>())
      .def("backend", [](worker::WorkerService& w, const std::string& id) { return w.backend(id); }, py::return_value_policy::reference_internal);

  // ---------------------------------------------------------------- client
  using client::BlackbirdClient;
  using client::BlackbirdClientOptions;
  py::class_<BlackbirdClientOptions>(m, "BlackbirdClientOptions")
      .def(py::init([](std::string host, uint16_t port, int timeout_ms, size_t par, std::string node_id, bool session) {
             BlackbirdClientOptions o;
             o.keystone_host = std::move(host);
             o.keystone_port = port;
             o.rpc_timeout_ms = timeout_ms;
             o.io_parallelism = par;
             o.node_id = std::move(node_id);
             o.register_session = session;
             return o;
           }),
           py::arg("keystone_host") = "127.0.0.1", py::arg("keystone_port") = 9090, py::arg("rpc_timeout_ms") = 30000,
           py::arg("io_parallelism") = 4, py::arg("node_id") = "", py::arg("register_session") = false)
      .def_readwrite("keystone_host", &BlackbirdClientOptions::keystone_host)
      .def_readwrite("keystone_port", &BlackbirdClientOptions::keystone_port)
      .def_readwrite("keystone_endpoints", &BlackbirdClientOptions::keystone_endpoints)
      .def_readwrite("rpc_timeout_ms", &BlackbirdClientOptions::rpc_timeout_ms)
      .def_readwrite("io_parallelism", &BlackbirdClientOptions::io_parallelism)
      .def_readwrite("node_id", &BlackbirdClientOptions::node_id)
      .def_readwrite("enable_shm", &BlackbirdClientOptions::enable_shm)
      .def_readwrite("auth_token", &BlackbirdClientOptions::auth_token)
      .def_readwrite("encrypt_transport", &BlackbirdClientOptions::encrypt_transport)
      .def_readwrite("auth_token_ro", &BlackbirdClientOptions::auth_token_ro)
      .def_readwrite("tenant", &BlackbirdClientOptions::tenant)
      .def_readwrite("tenant_secret", &BlackbirdClientOptions::tenant_secret);
  py::class_<BlackbirdClient, std::shared_ptr<BlackbirdClient>>(m, "BlackbirdClient")
      .def(py::init<BlackbirdClientOptions>(), py::arg("options") = BlackbirdClientOptions{})
      .def(py::init<std::shared_ptr<rpc::KeystoneApi>, BlackbirdClientOptions>(), py::arg("keystone"), py::arg("options") = BlackbirdClientOptions{})
      .def("connect", &BlackbirdClient::connect, py::call_guard<py::gil_scoped_release>())
      .def("connected", &BlackbirdClient::connected)
      .def_property_readonly("session_id", &BlackbirdClient::session_id)
      .def("object_exists", [](BlackbirdClient& c, const std::string& k) { return unwrap(c.object_exists(k)); }, py::call_guard<py::gil_scoped_release>())
      .def("get_workers", [](BlackbirdClient& c, const std::string& k) { return unwrap(c.get_workers(k)); }, py::call_guard<py::gil_scoped_release>())
      .def("put", [](BlackbirdClient& c, const std::string& key, py::buffer data, const WorkerConfig& cfg) {
        py::buffer_info i = data.request();
        py::gil_scoped_release rel;
        return c.put(key, static_cast<const uint8_t*>(i.ptr), static_cast<size_t>(i.size * i.itemsize), cfg);
      }, py::arg("key"), py::arg("data"), py::arg("config") = WorkerConfig{})
      .def("get", [](BlackbirdClient& c, const std::string& key) {
        Result<std::vector<uint8_t>> r = ErrorCode::INTERNAL_ERROR;
        {
          py::gil_scoped_release rel;
          r = c.get(key);
        }
        if (!r.ok()) throw BlackbirdError(r.error());
        return py::bytes(reinterpret_cast<const char*>(r.value().data()), r.value().size());
      })
      .def("remove", &BlackbirdClient::remove, py::call_guard<py::gil_scoped_release>())
      .def("migrate", &BlackbirdClient::migrate, py::call_guard<py::gil_scoped_release>())
      .def("batch_put_device_fp8",
           [](BlackbirdClient& c, const std::vector<ObjectKey>& keys, const std::vector<uintptr_t>& ptrs, const std::vector<uint64_t>& n_elems,
              const WorkerConfig& cfg, uintptr_t stream) {
             std::vector<const void*> p;
             for (auto v : ptrs) p.push_back(reinterpret_cast<const void*>(v));
             py::gil_scoped_release rel;
             return c.batch_put_device_fp8(keys, p, n_elems, cfg, reinterpret_cast<void*>(stream));
           },
           py::arg("keys"), py::arg("bf16_ptrs"), py::arg("n_elems"), py::arg("config"), py::arg("stream") = 0)
      .def("batch_get_device_fp8",
           [](BlackbirdClient& c, const std::vector<ObjectKey>& keys, const std::vector<uintptr_t>& ptrs, const std::vector<uint64_t>& n_elems,
              uintptr_t stream) {
             std::vector<void*> p;
             for (auto v : ptrs) p.push_back(reinterpret_cast<void*>(v));
             py::gil_scoped_release rel;
             return c.batch_get_device_fp8(keys, p, n_elems, reinterpret_cast<void*>(stream));
           },
           py::arg("keys"), py::arg("bf16_ptrs"), py::arg("n_elems"), py::arg("stream") = 0)
      .def("device_fp8_eligible", &BlackbirdClient::device_fp8_eligible)
      .def("batch_put", [](BlackbirdClient& c, const std::vector<std::string>& keys, const std::vector<py::buffer>& data, const WorkerConfig& cfg) {
        std::vector<const uint8_t*> ptrs;
        std::vector<size_t> sizes;
        std::vector<py::buffer_info> infos;
        for (const auto& b : data) infos.push_back(b.request());
        for (const auto& i : infos) {
          ptrs.push_back(static_cast<const uint8_t*>(i.ptr));
          sizes.push_back(static_cast<size_t>(i.size * i.itemsize));
        }
        py::gil_scoped_release rel;
        return c.batch_put(keys, ptrs, sizes, cfg);
      }, py::arg("keys"), py::arg("data"), py::arg("config") = WorkerConfig{})
      .def("batch_get", [](BlackbirdClient& c, const std::vector<std::string>& keys) {
        std::vector<Result<std::vector<uint8_t>>> r;
        {
          py::gil_scoped_release rel;
          r = c.batch_get(keys);
        }
        py::list out;
        for (const auto& e : r)
          out.append(py::make_tuple(e.error(), e.ok() ? py::object(py::bytes(reinterpret_cast<const char*>(e.value().data()), e.value().size()))
                                                      : py::object(py::none())));
        return out;
      })
      .def("batch_remove", [](BlackbirdClient& c, const std::vector<std::string>& keys) { return ecs_to_py(nogil([&] { return c.batch_remove(keys); })); })
      .def("batch_exists", [](BlackbirdClient& c, const std::vector<std::string>& keys) {
        return results_to_py(nogil([&] { return c.batch_exists(keys); }), [](bool b) { return py::bool_(b); });
      })
      .def("batch_put_device", [](BlackbirdClient& c, const std::vector<std::string>& keys, const std::vector<uintptr_t>& ptrs,
                                  const std::vector<size_t>& sizes, const WorkerConfig& cfg, uintptr_t stream) {
        std::vector<const void*> p;
        p.reserve(ptrs.size());
        for (auto v : ptrs) p.push_back(reinterpret_cast<const void*>(v));
        return ecs_to_py(nogil([&] { return c.batch_put_device(keys, p, sizes, cfg, reinterpret_cast<void*>(stream)); }));
      }, py::arg("keys"), py::arg("dev_ptrs"), py::arg("sizes"), py::arg("config") = WorkerConfig{}, py::arg("stream") = 0)
      .def("batch_get_device", [](BlackbirdClient& c, const std::vector<std::string>& keys, const std::vector<uintptr_t>& ptrs,
                                  const std::vector<size_t>& caps, uintptr_t stream) {
        std::vector<void*> p;
        for (auto v : ptrs) p.push_back(reinterpret_cast<void*>(v));
        std::vector<size_t> sizes;
        std::vector<ErrorCode> ecs;
        {
          py::gil_scoped_release rel;
          ecs = c.batch_get_device(keys, p, caps, reinterpret_cast<void*>(stream), &sizes);
        }
        return py::make_tuple(ecs_to_py(ecs), sizes);
      }, py::arg("keys"), py::arg("dev_ptrs"), py::arg("capacity"), py::arg("stream") = 0)
      .def("batch_put_device_gather", [](BlackbirdClient& c, const std::vector<std::string>& keys, const py::handle& segs,
                                         const std::vector<uint32_t>& seg_counts, const WorkerConfig& cfg, uintptr_t stream) {
        auto a = py_segments::read_segments(segs);
        std::vector<DeviceSegment> v(a.count);
        if (a.count) std::memcpy(v.data(), a.data, a.count * sizeof(DeviceSegment));
        return ecs_to_py(nogil([&] { return c.batch_put_device_gather(keys, v, seg_counts, cfg, reinterpret_cast<void*>(stream)); }));
      }, py::arg("keys"), py::arg("segs"), py::arg("seg_counts"), py::arg("config") = WorkerConfig{}, py::arg("stream") = 0,
         "Segmented put: object i is the concatenation of the next seg_counts[i] rows (device pointer, bytes) of the (S, 2) "
         "uint64 / int64 array `segs`.  Stored exactly as a contiguous put of that concatenation.")
      .def("batch_get_device_scatter", [](BlackbirdClient& c, const std::vector<std::string>& keys, const py::handle& segs,
                                          const std::vector<uint32_t>& seg_counts, uintptr_t stream) {
        auto a = py_segments::read_segments(segs);
        std::vector<DeviceSegment> v(a.count);
        if (a.count) std::memcpy(v.data(), a.data, a.count * sizeof(DeviceSegment));
        return ecs_to_py(nogil([&] { return c.batch_get_device_scatter(keys, v, seg_counts, reinterpret_cast<void*>(stream)); }));
      }, py::arg("keys"), py::arg("segs"), py::arg("seg_counts"), py::arg("stream") = 0,
         "Segmented get: object i is scattered over the next seg_counts[i] rows of `segs`; their lengths must add up to the "
         "stored size.")
      .def("cluster_stats", [](BlackbirdClient& c) { return unwrap(nogil([&] { return c.cluster_stats(); })); })
      .def("metrics_text", &BlackbirdClient::metrics_text)
      .def("set_device_pipeline_chunks", &BlackbirdClient::set_device_pipeline_chunks)
      .def("phase_summary", &BlackbirdClient::phase_summary, "histogram name -> [count, sum_us, p50_us, p99_us]")
      .def("keystone", [](BlackbirdClient& c) -> rpc::KeystoneApi& { return c.keystone(); }, py::return_value_policy::reference_internal);
}
