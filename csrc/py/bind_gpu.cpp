// Bindings for the sm_100a data plane: XferEngine (fused batched transfer), comparators and
// device helpers.  Pointers cross the boundary as integers (tensor.data_ptr()), streams as
// integers (torch.cuda.current_stream().cuda_stream).
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include "client/blackbird_client.h"
#include "fabric/gpu_fabric.h"
#include "fabric/xfer_engine.h"
#include "kernels/xfer.h"
#include "py/segments.h"

#include <deque>

namespace py = pybind11;
using namespace bb;
using namespace bb::gpu;

namespace {
void check(ErrorCode ec, const char* what) {
  if (ec != ErrorCode::OK) throw std::runtime_error(std::string(what) + ": " + std::string(to_string(ec)));
}
void check_cuda(int rc, const char* what) {
  if (rc != 0) throw std::runtime_error(std::string(what) + ": CUDA error " + std::to_string(rc) + " " + cuda_error_string(rc));
}
// item tuple: (src | segments, dst | [dst...] | segments, nbytes, expect=0, flags=0).  `segments` = an (S, 2) array of
// (device pointer, bytes) rows (py/segments.h): a gathered source or a scattered destination.  `keep` holds the arrays
// until the batch is submitted (the engine copies the tables into its staging buffer).
XferItem to_item(const py::handle& h, std::deque<py_segments::SegmentArray>& keep) {
  py::tuple t = py::cast<py::tuple>(h);
  if (t.size() < 3) throw py::value_error("xfer item = (src|segments, dst|[dst..]|segments, nbytes[, expect[, flags]])");
  XferItem it;
  if (py_segments::is_segment_array(t[0])) {
    keep.push_back(py_segments::read_segments(t[0]));
    it.segs = keep.back().data;
    it.nsegs = static_cast<uint32_t>(keep.back().count);
    it.flags |= XFER_GATHER;
  } else {
    it.src = reinterpret_cast<const void*>(t[0].cast<uintptr_t>());
  }
  if (py_segments::is_segment_array(t[1])) {
    if (it.segs) throw py::value_error("an item gathers or scatters, not both");
    keep.push_back(py_segments::read_segments(t[1]));
    it.segs = keep.back().data;
    it.nsegs = static_cast<uint32_t>(keep.back().count);
    it.flags |= XFER_SCATTER;
    it.ndst = 1;
  } else if (py::isinstance<py::int_>(t[1])) {
    it.dst[0] = reinterpret_cast<void*>(t[1].cast<uintptr_t>());
    it.ndst = 1;
  } else {
    auto v = t[1].cast<std::vector<uintptr_t>>();
    if (v.empty() || v.size() > kMaxDst) throw py::value_error("1..3 destinations");
    it.ndst = static_cast<uint32_t>(v.size());
    for (size_t i = 0; i < v.size(); ++i) it.dst[i] = reinterpret_cast<void*>(v[i]);
  }
  it.nbytes = t[2].cast<uint64_t>();
  if (t.size() > 3) it.expect = t[3].cast<uint64_t>();
  if (t.size() > 4) it.flags |= t[4].cast<uint32_t>();
  return it;
}
}  // namespace

void bind_gpu(py::module_& m) {
  m.attr("TILE_BYTES") = kTileBytes;
  m.attr("XFER_VERIFY") = static_cast<uint32_t>(XFER_VERIFY);
  m.attr("XFER_MULTIMEM") = static_cast<uint32_t>(XFER_MULTIMEM);
  m.attr("XFER_GATHER") = static_cast<uint32_t>(XFER_GATHER);
  m.attr("XFER_SCATTER") = static_cast<uint32_t>(XFER_SCATTER);
  m.def("cuda_device_count", [] {
    int n = 0;
    device_count(&n);
    return n;
  });

  py::class_<XferEngine>(m, "XferEngine")
      .def(py::init([](int device, uint32_t max_items, int slots) {
             auto r = XferEngine::create(device, max_items, slots);
             if (!r.ok()) throw std::runtime_error("XferEngine.create: " + std::string(to_string(r.error())));
             return std::move(r.value());
           }),
           py::arg("device") = 0, py::arg("max_items") = 1u << 16, py::arg("slots") = 4)
      .def("run",
           [](XferEngine& e, const py::list& items, ChecksumAlgo algo, uintptr_t stream, bool debug) {
             std::vector<XferItem> v;
             std::deque<py_segments::SegmentArray> keep;
             v.reserve(items.size());
             for (auto h : items) v.push_back(to_item(h, keep));
             XferResult res;
             {
               py::gil_scoped_release rel;
               auto t = e.submit(v, algo, reinterpret_cast<void*>(stream), debug);
               if (!t.ok()) check(t.error(), "XferEngine.submit");
               check(e.wait(t.value(), &res), "XferEngine.wait");
             }
             return py::make_tuple(res.digest, res.status, res.device_ms);
           },
           py::arg("items"), py::arg("algo") = ChecksumAlgo::BBH64, py::arg("stream") = 0, py::arg("debug") = false,
           "Runs one fused batch; returns (digests, status, device_ms).")
      .def("run_fp8",
           [](XferEngine& e, const py::list& items, bool unpack, uintptr_t stream) {
             std::vector<gpu::Fp8Item> v;
             for (auto h : items) {
               auto t = h.cast<py::tuple>();
               if (t.size() < 3) throw py::value_error("fp8 item = (bf16, packed|[packed..], n_elems[, expect])");
               gpu::Fp8Item it;
               it.wide = reinterpret_cast<void*>(t[0].cast<uintptr_t>());
               if (py::isinstance<py::int_>(t[1])) {
                 it.packed = reinterpret_cast<void*>(t[1].cast<uintptr_t>());
               } else {
                 auto p = t[1].cast<std::vector<uintptr_t>>();
                 if (p.empty() || p.size() > kMaxDst) throw py::value_error("1..3 packed replicas");
                 if (unpack && p.size() > 1) throw py::value_error("a get reads one packed copy");
                 it.packed = reinterpret_cast<void*>(p[0]);
                 for (size_t r = 1; r < p.size(); ++r) it.more_packed[r - 1] = reinterpret_cast<void*>(p[r]);
                 it.nreplicas = static_cast<uint32_t>(p.size());
               }
               it.n_elems = t[2].cast<uint64_t>();
               if (t.size() > 3) it.expect = t[3].cast<uint64_t>(), it.verify = true;
               v.push_back(it);
             }
             XferResult res;
             {
               py::gil_scoped_release rel;
               check(e.run_fp8(v, unpack, reinterpret_cast<void*>(stream), &res), "XferEngine.run_fp8");
             }
             return py::make_tuple(res.digest, res.status, res.device_ms);
           },
           py::arg("items"), py::arg("unpack"), py::arg("stream") = 0,
           "Fused MXFP8 put (unpack=False: bf16 -> packed slab object) or get (unpack=True); items = (bf16_ptr, packed_ptr | "
           "[packed_ptr, ...], n_elems[, expected_digest]); a put writes every listed replica (1..3), a get reads one; "
           "returns (digests of the packed objects, status, device_ms).")
      .def_static("fp8_eligible", &XferEngine::fp8_eligible)
      .def("submit",
           [](XferEngine& e, const py::list& items, ChecksumAlgo algo, uintptr_t stream) {
             std::vector<XferItem> v;
             std::deque<py_segments::SegmentArray> keep;
             v.reserve(items.size());
             for (auto h : items) v.push_back(to_item(h, keep));
             auto t = e.submit(v, algo, reinterpret_cast<void*>(stream));
             if (!t.ok()) check(t.error(), "XferEngine.submit");
             return t.value();
           },
           py::arg("items"), py::arg("algo") = ChecksumAlgo::BBH64, py::arg("stream") = 0)
      .def("wait",
           [](XferEngine& e, uint64_t ticket) {
             XferResult res;
             {
               py::gil_scoped_release rel;
               check(e.wait(ticket, &res), "XferEngine.wait");
             }
             return py::make_tuple(res.digest, res.status, res.device_ms);
           })
      .def("debug_accumulators", [](XferEngine& e) { return e.debug_accumulators(); })
      .def("set_max_ctas", &XferEngine::set_max_ctas)
      .def("set_small_path", &XferEngine::set_small_path)
      .def("set_flag_completion", &XferEngine::set_flag_completion)
      .def("set_mailbox", &XferEngine::set_mailbox)
      .def_property_readonly("mailbox_requests", &XferEngine::mailbox_requests)
      .def_property_readonly("mailbox_launches", &XferEngine::mailbox_launches)
      .def_property_readonly("small_launches", &XferEngine::small_launches)
      .def("set_tile_trace", &XferEngine::set_tile_trace)
      .def("tile_trace", [](XferEngine& e) { return e.tile_trace(); }, "[tile][4] globaltimer ns: load issued, landed, store issued, slot released")
      .def_property_readonly("launches", &XferEngine::launches)
      .def_property_readonly("device", &XferEngine::device);

  m.def("copy_simt", [](uintptr_t dst, uintptr_t src, uint64_t n, uintptr_t stream) {
    check_cuda(launch_copy_simt(reinterpret_cast<void*>(dst), reinterpret_cast<const void*>(src), n,
                                reinterpret_cast<void*>(stream)), "copy_simt");
  }, py::arg("dst"), py::arg("src"), py::arg("nbytes"), py::arg("stream") = 0);
  m.def("crc32c_device", [](uintptr_t data, uint64_t n, uintptr_t out, uintptr_t scratch, uintptr_t stream) {
    check_cuda(launch_crc32c_simt(reinterpret_cast<const void*>(data), n, reinterpret_cast<uint32_t*>(out),
                                  reinterpret_cast<uint32_t*>(scratch), reinterpret_cast<void*>(stream)), "crc32c_device");
  }, py::arg("data"), py::arg("nbytes"), py::arg("out"), py::arg("scratch"), py::arg("stream") = 0,
     "Stand-alone CRC32C; scratch needs 4*ceil(nbytes/512) bytes.");
  m.def("fill", [](uintptr_t dst, uint64_t n, uint32_t v, uintptr_t stream) {
    check_cuda(launch_fill(reinterpret_cast<void*>(dst), n, v, reinterpret_cast<void*>(stream)), "fill");
  }, py::arg("dst"), py::arg("nbytes"), py::arg("value") = 0, py::arg("stream") = 0);
  m.def("random_fill", [](uintptr_t dst, uint64_t n, uint64_t seed, uintptr_t stream) {
    check_cuda(launch_random_fill(reinterpret_cast<void*>(dst), n, seed, reinterpret_cast<void*>(stream)), "random_fill");
  }, py::arg("dst"), py::arg("nbytes"), py::arg("seed") = 1, py::arg("stream") = 0);
  m.def("memcpy_peer_async", [](uintptr_t dst, int dst_dev, uintptr_t src, int src_dev, uint64_t n, uintptr_t stream) {
    check_cuda(device_memcpy_peer_async(reinterpret_cast<void*>(dst), dst_dev, reinterpret_cast<const void*>(src), src_dev, n,
                                        reinterpret_cast<void*>(stream)), "memcpy_peer_async");
  }, py::arg("dst"), py::arg("dst_device"), py::arg("src"), py::arg("src_device"), py::arg("nbytes"), py::arg("stream") = 0,
     "cudaMemcpyPeerAsync (copy engines): the naive P2P comparator of BASELINE.md section 4.");
  m.def("enable_peer_access", [](int device, int peer) { check_cuda(device_enable_peer_access(device, peer), "enable_peer_access"); });
  m.def("xfer_smem_bytes", [] { return xfer_smem_bytes(ALGO_BBH64); });
  m.def("mxfp8_pack", [](uintptr_t src, uint64_t n, uintptr_t dst, uintptr_t stream) {
    check_cuda(launch_mxfp8_pack(reinterpret_cast<const void*>(src), n, reinterpret_cast<void*>(dst), reinterpret_cast<void*>(stream)), "mxfp8_pack");
  }, py::arg("src_bf16"), py::arg("n_elems"), py::arg("dst_packed"), py::arg("stream") = 0);
  m.def("mxfp8_unpack", [](uintptr_t src, uint64_t n, uintptr_t dst, uintptr_t stream) {
    check_cuda(launch_mxfp8_unpack(reinterpret_cast<const void*>(src), n, reinterpret_cast<void*>(dst), reinterpret_cast<void*>(stream)), "mxfp8_unpack");
  }, py::arg("src_packed"), py::arg("n_elems"), py::arg("dst_bf16"), py::arg("stream") = 0);

  // ---- fabric: GPU tier + device transport of the client SDK
  m.def("install_gpu_backend_factory", &install_gpu_backend_factory,
        "Registers the RAM_GPU storage tier (cudaMalloc slab + CUDA IPC export) with the worker.");
  py::class_<GpuFabric, std::shared_ptr<GpuFabric>>(m, "GpuFabric")
      .def(py::init([](int device, std::shared_ptr<rpc::KeystoneApi> ks) {
             auto f = GpuFabric::create(device, std::move(ks));
             if (!f.ok()) throw std::runtime_error("GpuFabric.create: " + std::string(to_string(f.error())));
             return f.value();
           }),
           py::arg("device"), py::arg("keystone"))
      .def("refresh_pools", &GpuFabric::refresh_pools, py::call_guard<py::gil_scoped_release>())
      .def("mapped_pools", &GpuFabric::mapped_pools)
      .def("mapped_host_pools", &GpuFabric::mapped_host_pools)
      .def_property_readonly("remaps", &GpuFabric::remaps)
      .def("metrics_text", &GpuFabric::metrics_text)
      .def("path_bytes", &GpuFabric::path_bytes, py::arg("put"), py::arg("path"), "path: 0 hbm, 1 nvlink, 2 pcie, 3 nvlink multicast")
      .def_property_readonly("launches", &GpuFabric::launches)
      .def_property_readonly("last_device_ms", &GpuFabric::last_device_ms)
      .def_property_readonly("total_device_ms", &GpuFabric::total_device_ms)
      .def("set_max_ctas", [](GpuFabric& f, int n) { f.engine().set_max_ctas(n); })
      .def("set_small_path", [](GpuFabric& f, bool on) { f.engine().set_small_path(on); })
      .def("set_flag_completion", [](GpuFabric& f, bool on) { f.engine().set_flag_completion(on); })
      .def("set_mailbox", [](GpuFabric& f, bool on) { f.engine().set_mailbox(on); })
      .def_property_readonly("mailbox_requests", [](GpuFabric& f) { return f.engine().mailbox_requests(); })
      .def_property_readonly("mailbox_launches", [](GpuFabric& f) { return f.engine().mailbox_launches(); })
      .def_property_readonly("small_launches", [](GpuFabric& f) { return f.engine().small_launches(); })
      .def("set_tile_trace", [](GpuFabric& f, bool on) { f.engine().set_tile_trace(on); })
      .def("tile_trace", [](GpuFabric& f) { return f.engine().tile_trace(); })
      .def("set_arena", &GpuFabric::set_arena)
      .def_property_readonly("multicast_puts", &GpuFabric::multicast_puts);
  py::class_<NvlsArena, std::shared_ptr<NvlsArena>>(m, "NvlsArena")
      .def(py::init<int, int, int, std::string, std::vector<std::vector<int>>, uint64_t>(), py::arg("device"), py::arg("rank"), py::arg("world"),
           py::arg("tag"), py::arg("groups"), py::arg("arena_bytes"))
      .def_static("supported", &NvlsArena::supported)
      .def("phase1_create", &NvlsArena::phase1_create, py::call_guard<py::gil_scoped_release>())
      .def("phase2_join", &NvlsArena::phase2_join, py::call_guard<py::gil_scoped_release>())
      .def("phase3_bind", &NvlsArena::phase3_bind, py::call_guard<py::gil_scoped_release>())
      .def("phase4_map_peers", &NvlsArena::phase4_map_peers, py::call_guard<py::gil_scoped_release>())
      .def("num_groups", &NvlsArena::num_groups)
      .def("members", &NvlsArena::members)
      .def("member_of", &NvlsArena::member_of)
      .def_property_readonly("arena_bytes", &NvlsArena::arena_bytes)
      .def("mc_ptr", [](NvlsArena& a, size_t g) { return reinterpret_cast<uintptr_t>(a.mc_ptr(g)); })
      .def("peer_ptr", [](NvlsArena& a, size_t g, int r) { return reinterpret_cast<uintptr_t>(a.peer_ptr(g, r)); })
      .def_static("pool_id", &NvlsArena::pool_id)
      .def_static("domain", &NvlsArena::domain)
      .def_property_readonly("last_error", &NvlsArena::last_error);
  m.def("attach_fabric", [](client::BlackbirdClient& c, std::shared_ptr<GpuFabric> f) { c.set_device_transport(std::move(f)); });
}
