"""End-to-end on CPU (BASELINE config #1): in-process Keystone + 2 workers over loopback TCP,
put/get/exists/remove of 1 KB objects; RPC façade (all methods), HTTP /metrics, worker
registration + heartbeats through the coordination store, failure detection, replica
fail-over, checksum enforcement, striping, batch API, multi-tier workers, config files."""
import os
import threading
import time

import pytest

from blackbird_b200.parallel import LocalCluster


@pytest.fixture
def cluster(bb):
    with LocalCluster("e2e", n_workers=2, pool_bytes=64 << 20) as c:
        yield c


def test_config1_put_get_exists_remove_1kb(bb, cluster):
    cl = cluster.client()
    data = os.urandom(1024)
    cfg = bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1)
    assert cl.object_exists("k") is False
    assert cl.put("k", data, cfg) == bb.ErrorCode.OK
    assert cl.object_exists("k") is True and cl.get("k") == data
    copies = cl.get_workers("k")
    sh = copies[0].shards[0]
    assert sh.length == 1024 and sh.checksum == bb.bbh64(data) and sh.storage_class == bb.StorageClass.RAM_CPU
    assert cl.put("k", data, cfg) == bb.ErrorCode.OBJECT_ALREADY_EXISTS
    assert cl.remove("k") == bb.ErrorCode.OK and cl.object_exists("k") is False
    with pytest.raises(bb.BlackbirdError) as e:
        cl.get("k")
    assert e.value.code == bb.ErrorCode.OBJECT_NOT_FOUND
    st = cl.cluster_stats()
    assert st.total_workers == 2 and st.total_memory_pools == 2 and st.total_objects == 0 and st.used_capacity == 0


def test_workers_register_through_coordination_schema(bb, cluster):
    keys = [k for k, *_ in cluster.coord.store().get_with_prefix("/blackbird/clusters/e2e/")]
    assert "/blackbird/clusters/e2e/workers/worker-0" in keys
    assert "/blackbird/clusters/e2e/workers/worker-0/memory_pools/pool-0" in keys
    assert "/blackbird/clusters/e2e/heartbeat/worker-1" in keys
    assert cluster.coord.discover_service("blackbird-keystone") == [cluster.cfg.listen_address]
    pool = bb.MemoryPool.from_json(cluster.coord.store().get("/blackbird/clusters/e2e/workers/worker-0/memory_pools/pool-0").decode())
    assert pool.worker_id == "worker-0" and pool.size == 64 << 20 and pool.ucx_endpoint == cluster.workers[0].data_endpoint()
    assert len(pool.ucx_rkey_hex) == 8  # fixed-width hex (reference bug #7: unpadded, colon separated)
    info = {w["worker_id"]: w for w in cluster.keystone.get_workers_info()}
    assert info["worker-0"]["pools"] == ["pool-0"]


def test_striping_replication_and_checksums_over_tcp(bb, cluster):
    cl = cluster.client(io_parallelism=4)
    data = os.urandom(3 * (1 << 20) + 12345)
    for algo in (bb.ChecksumAlgo.CRC32C, bb.ChecksumAlgo.BBH64, bb.ChecksumAlgo.NONE):
        key = f"striped-{algo.name}"
        cfg = bb.WorkerConfig(replication_factor=2, max_workers_per_copy=2, checksum=algo, min_shard_size=4096)
        assert cl.put(key, data, cfg) == bb.ErrorCode.OK
        copies = cl.get_workers(key)
        assert len(copies) == 2 and sum(s.length for s in copies[0].shards) == len(data)
        if algo == bb.ChecksumAlgo.CRC32C:
            off = 0
            for s in copies[0].shards:
                assert s.checksum == bb.crc32c(data[off:off + s.length])
                off += s.length
        assert cl.get(key) == data


def test_corruption_is_detected_and_reads_fail_over_to_replica(bb, cluster):
    cl = cluster.client()
    data = os.urandom(200000)
    assert cl.put("r2", data, bb.WorkerConfig(replication_factor=2, max_workers_per_copy=1)) == bb.ErrorCode.OK
    copies = cl.get_workers("r2")
    victim = copies[0].shards[0]
    worker = next(w for w in cluster.workers if w.data_endpoint() == f"{victim.endpoint.ip}:{victim.endpoint.port}")
    base = worker.backend(victim.pool_id).get_base_address()
    worker.backend(victim.pool_id).write(victim.offset - base + 1000, b"\x00" * 64)  # silent corruption of copy 0
    assert cl.get("r2") == data  # served from the intact replica
    assert "bb_client_replica_failover_total 1" in cl.metrics_text() and "bb_client_checksum_mismatch_total 1" in cl.metrics_text()
    cl.put("r1", data, bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1))
    s1 = cl.get_workers("r1")[0].shards[0]
    w1 = next(w for w in cluster.workers if w.data_endpoint() == f"{s1.endpoint.ip}:{s1.endpoint.port}")
    w1.backend(s1.pool_id).write(s1.offset - w1.backend(s1.pool_id).get_base_address(), b"\xff" * 8)
    with pytest.raises(bb.BlackbirdError) as e:
        cl.get("r1")
    assert e.value.code == bb.ErrorCode.CHECKSUM_MISMATCH  # the code exists in the reference but nothing produces it


def test_batch_put_get_remove(bb, cluster):
    cl = cluster.client()
    keys = [f"b{i}" for i in range(50)]
    blobs = [os.urandom(1024 + i) for i in range(50)]
    cfg = bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1)
    assert cl.batch_put(keys, blobs, cfg) == [bb.ErrorCode.OK] * 50
    assert cl.batch_put(keys[:2], blobs[:2], cfg) == [bb.ErrorCode.OBJECT_ALREADY_EXISTS] * 2
    res = cl.batch_get(keys + ["missing"])
    assert [r[1] for r in res[:50]] == blobs and res[50][0] == bb.ErrorCode.OBJECT_NOT_FOUND
    assert [v for _, v in cl.batch_exists(keys[:3] + ["missing"])] == [True, True, True, False]
    assert cl.batch_remove(keys) == [bb.ErrorCode.OK] * 50
    assert cluster.keystone.get_cluster_stats().used_capacity == 0


def test_rpc_facade_all_methods_and_http(bb, cluster):
    api = bb.KeystoneRpcClient()
    assert api.connect("127.0.0.1", cluster.rpc.rpc_port) == bb.ErrorCode.OK
    cfg = bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1)
    v0 = api.get_view_version()
    copies = api.put_start("rpc-k", 5000, cfg)
    assert copies[0].shards[0].length == 5000 and copies[0].shards[0].endpoint.port > 0
    assert api.put_complete("rpc-k", [[42]]) == bb.ErrorCode.OK
    assert api.object_exists("rpc-k") is True and api.get_workers("rpc-k")[0].shards[0].checksum == 42
    assert api.get_view_version() > v0
    res = api.batch_put_start(["x1", "x2", "rpc-k"], [10, 20, 30], cfg)
    assert [r[0] for r in res] == [bb.ErrorCode.OK, bb.ErrorCode.OK, bb.ErrorCode.OBJECT_ALREADY_EXISTS]
    assert api.batch_put_complete(["x1"]) == [bb.ErrorCode.OK]
    assert api.batch_put_cancel(["x2", "nope"]) == [bb.ErrorCode.OK, bb.ErrorCode.OBJECT_NOT_FOUND]
    assert [r[1] for r in api.batch_object_exists(["x1", "x2"])] == [True, False]
    assert api.batch_get_workers(["x1", "x2"])[1][0] == bb.ErrorCode.OBJECT_NOT_FOUND
    st = api.get_cluster_stats()
    assert st.total_objects == 2 and st.total_workers == 2
    assert {p.id for p in api.get_memory_pools()} == {"pool-0", "pool-1"}
    cid = api.client_register("node-9")
    assert api.client_ping(cid) >= 1
    assert api.batch_remove_object(["x1"]) == [bb.ErrorCode.OK]
    assert api.remove_object("rpc-k") == bb.ErrorCode.OK and api.remove_all_objects() == 0
    assert api.put_cancel("nope") == bb.ErrorCode.OBJECT_NOT_FOUND
    status, body = bb.http_get("127.0.0.1", cluster.rpc.http_port, "/metrics")
    assert status == 200 and "bb_put_start_total" in body and "# TYPE bb_objects gauge" in body
    status, body = bb.http_get("127.0.0.1", cluster.rpc.http_port, "/healthz")
    assert status == 200 and body.startswith("ok")
    status, body = bb.http_get("127.0.0.1", cluster.rpc.http_port, "/stats")
    assert status == 200 and bb.parse_json(body)["cluster"]["total_workers"] == 2
    assert bb.http_get("127.0.0.1", cluster.rpc.http_port, "/nope")[0] == 404
    assert cluster.rpc.requests_served > 15


def test_many_concurrent_rpc_clients(bb, cluster):
    errs = []

    def run(t):
        try:
            cl = cluster.client()
            cfg = bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1)
            for i in range(40):
                d = os.urandom(777)
                assert cl.put(f"c{t}/{i}", d, cfg) == bb.ErrorCode.OK
                assert cl.get(f"c{t}/{i}") == d
                assert cl.remove(f"c{t}/{i}") == bb.ErrorCode.OK
        except Exception as ex:  # noqa: BLE001
            errs.append(repr(ex))

    ts = [threading.Thread(target=run, args=(t,)) for t in range(8)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errs, errs[:2]


def test_failure_detection_lease_expiry_removes_worker_and_objects(bb):
    with LocalCluster("fd", n_workers=2, pool_bytes=8 << 20, lease_ttl_sec=2, heartbeat_interval_sec=1) as c:
        cl = c.client()
        data = os.urandom(4096)
        assert cl.put("both", data, bb.WorkerConfig(replication_factor=2, max_workers_per_copy=1)) == bb.ErrorCode.OK
        assert cl.put("only0", data, bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1, preferred_node="node-0")) == bb.ErrorCode.OK
        c.workers[0].inject_fault("drop_heartbeat")  # worker-0 hangs: stops refreshing its lease
        store = c.coord.store()
        deadline = time.time() + 10
        while c.keystone.get_cluster_stats().total_workers == 2 and time.time() < deadline:
            time.sleep(0.1)
        store.flush_events()
        st = c.keystone.get_cluster_stats()
        assert st.total_workers == 1 and st.total_memory_pools == 1
        assert store.get("/blackbird/clusters/fd/workers/worker-0") is None  # keystone cleaned the registry
        assert cl.get("both") == data  # surviving replica
        with pytest.raises(bb.BlackbirdError):
            cl.get("only0")  # its only copy died with the worker
        assert "bb_worker_deaths_total 1" in c.keystone.metrics_text()
        # new puts avoid the dead worker
        assert cl.put("after", data, bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1)) == bb.ErrorCode.OK
        assert cl.get_workers("after")[0].shards[0].worker_id == "worker-1"


def test_multi_tier_worker_and_class_preference(bb, tmp_path):
    with LocalCluster("tiers", n_workers=0) as c:
        c.add_worker("w-tiers", "node-t", [("dram", bb.StorageClass.RAM_CPU, 8 << 20, ""), ("nvme", bb.StorageClass.NVME, 32 << 20, str(tmp_path)),
                                            ("cxl", bb.StorageClass.CXL_MEMORY, 8 << 20, ""), ("hdd", bb.StorageClass.HDD, 16 << 20, str(tmp_path))])
        cl = c.client()
        data = os.urandom(300000)
        for name, sc in [("dram", bb.StorageClass.RAM_CPU), ("nvme", bb.StorageClass.NVME), ("cxl", bb.StorageClass.CXL_MEMORY), ("hdd", bb.StorageClass.HDD)]:
            cfg = bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1, preferred_classes=[sc], checksum=bb.ChecksumAlgo.CRC32C)
            assert cl.put(f"on-{name}", data, cfg) == bb.ErrorCode.OK
            sh = cl.get_workers(f"on-{name}")[0].shards[0]
            assert sh.pool_id == name and sh.storage_class == sc
            assert cl.get(f"on-{name}") == data
        stats = c.workers[0].get_stats()
        assert {p["pool_id"] for p in stats["pools"]} == {"dram", "nvme", "cxl", "hdd"} and stats["requests_served"] >= 8
        assert all(p["bytes_written"] >= 300000 for p in stats["pools"])


def test_config_files_parse(bb, tmp_path):
    reference_configs = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_configs")
    ks = bb.KeystoneConfig.from_yaml(os.path.join(reference_configs, "keystone.yaml"))  # reference sample parses unchanged
    assert ks.cluster_id == "blackbird_cluster" and ks.etcd_endpoints == "localhost:2379" and ks.high_watermark == 0.8
    assert ks.client_ttl_sec == 300 and ks.max_replicas == 3 and ks.log_level == "INFO"
    wc = bb.WorkerServiceConfig.from_yaml(os.path.join(reference_configs, "worker.yaml"))
    assert wc.worker_id == "worker-1" and wc.interconnects == ["rdma", "tcp"] and wc.heartbeat_interval_sec == 5
    assert wc.storage_pools[0].pool_id == "ram_pool_0" and wc.storage_pools[0].size_bytes == 2 << 30
    for name in ("keystone.yaml", "worker.yaml", "gpu_worker.yaml", "tiered_worker.yaml"):
        path = os.path.join(os.path.dirname(os.path.dirname(__file__)), "configs", name)
        (bb.KeystoneConfig.from_yaml if name.startswith("keystone") else bb.WorkerServiceConfig.from_yaml)(path)
    bad = tmp_path / "bad.yaml"
    bad.write_text("keystone:\n  cluster_id: x\n  high_watermark: 1.5\n")
    with pytest.raises(RuntimeError, match="high_watermark"):
        bb.KeystoneConfig.from_yaml(str(bad))
    bad.write_text("worker:\n  worker_id: w\n  lease_ttl_sec: 5\n  heartbeat_interval_sec: 9\n")
    with pytest.raises(RuntimeError, match="heartbeat_interval_sec"):
        bb.WorkerServiceConfig.from_yaml(str(bad))


def test_config4_tier_spill_dram_to_nvme_with_ttl_and_soft_pin(bb, tmp_path):
    """BASELINE config #4 on host tiers: watermark eviction demotes LRU objects DRAM -> NVMe through the
    worker's data path (real bytes, digests re-verified), soft-pinned objects stay, TTL'd objects expire."""
    kc = bb.KeystoneConfig()
    kc.high_watermark = 0.5
    kc.eviction_ratio = 0.5
    kc.gc_interval_sec = 3600
    kc.health_check_interval_sec = 3600
    with LocalCluster("spill", n_workers=0, keystone_cfg=kc) as c:
        c.add_worker("w0", "node-0", [("dram", bb.StorageClass.RAM_CPU, 8 << 20, ""), ("nvme", bb.StorageClass.NVME, 64 << 20, str(tmp_path))])
        c.keystone.install_data_server_mover()
        cl = c.client()
        blobs = {}
        ram = dict(replication_factor=1, max_workers_per_copy=1, preferred_classes=[bb.StorageClass.RAM_CPU], checksum=bb.ChecksumAlgo.CRC32C)
        for i in range(5):
            blobs[f"o{i}"] = os.urandom(1 << 20)
            assert cl.put(f"o{i}", blobs[f"o{i}"], bb.WorkerConfig(ttl_ms=0, **ram)) == bb.ErrorCode.OK
            time.sleep(0.01)
        blobs["pinned"] = os.urandom(1 << 20)
        assert cl.put("pinned", blobs["pinned"], bb.WorkerConfig(ttl_ms=0, enable_soft_pin=True, **ram)) == bb.ErrorCode.OK
        blobs["ttl"] = os.urandom(1 << 20)
        assert cl.put("ttl", blobs["ttl"], bb.WorkerConfig(ttl_ms=1500, **ram)) == bb.ErrorCode.OK  # long enough for a sanitizer build to get through the reads below
        assert c.keystone.tier_utilization(bb.StorageClass.RAM_CPU) > 0.8
        cl.get("o0")  # o0 becomes most recently used
        n = c.keystone.run_eviction_once()
        assert n >= 3
        tiers = {k: cl.get_workers(k)[0].shards[0].storage_class for k in list(blobs)}
        assert tiers["pinned"] == bb.StorageClass.RAM_CPU and tiers["o0"] == bb.StorageClass.RAM_CPU  # pin + LRU respected
        assert tiers["o1"] == bb.StorageClass.NVME and tiers["o2"] == bb.StorageClass.NVME
        for k, v in blobs.items():
            assert cl.get(k) == v, k  # demoted objects read back bit-exact from NVMe (CRC verified)
        sh = cl.get_workers("o1")[0].shards[0]
        assert sh.checksum == bb.crc32c(blobs["o1"]) and sh.location["kind"] == "file"
        assert c.keystone.tier_utilization(bb.StorageClass.RAM_CPU) <= 0.55
        text = c.keystone.metrics_text()
        assert "bb_demotions_total" in text and "bb_evictions_total" not in text  # nothing was dropped
        time.sleep(1.6)
        assert c.keystone.run_gc_once() == 1 and cl.object_exists("ttl") is False
        stats = c.workers[0].get_stats()
        nv = next(p for p in stats["pools"] if p["pool_id"] == "nvme")
        assert nv["bytes_written"] >= 3 << 20


def test_explicit_migrate_promotes_and_demotes_across_tiers(bb, tmp_path):
    """migrate_object: every copy moves to the target tier through the workers' D_COPY path, digests are
    re-checked by the mover, old extents are freed, and the object stays readable throughout."""
    with LocalCluster("migrate", n_workers=0) as c:
        c.add_worker("w0", "node-0", [("dram", bb.StorageClass.RAM_CPU, 16 << 20, ""), ("nvme", bb.StorageClass.NVME, 64 << 20, str(tmp_path))])
        c.keystone.install_data_server_mover()
        cl = c.client()
        blob = os.urandom(3 << 20)
        cfg = bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1, ttl_ms=0, preferred_classes=[bb.StorageClass.RAM_CPU], checksum=bb.ChecksumAlgo.CRC32C)
        assert cl.put("m", blob, cfg) == bb.ErrorCode.OK
        used_before = c.keystone.tier_utilization(bb.StorageClass.RAM_CPU)
        assert cl.migrate("m", bb.StorageClass.NVME) == bb.ErrorCode.OK
        sh = cl.get_workers("m")[0].shards[0]
        assert sh.storage_class == bb.StorageClass.NVME and sh.checksum == bb.crc32c(blob)
        assert c.keystone.tier_utilization(bb.StorageClass.RAM_CPU) < used_before  # DRAM extent released
        assert cl.get("m") == blob
        assert cl.migrate("m", bb.StorageClass.NVME) == bb.ErrorCode.OK  # already there: no-op
        assert cl.migrate("m", bb.StorageClass.RAM_CPU) == bb.ErrorCode.OK  # promotion
        assert cl.get_workers("m")[0].shards[0].storage_class == bb.StorageClass.RAM_CPU and cl.get("m") == blob
        assert cl.migrate("nope", bb.StorageClass.NVME) == bb.ErrorCode.OBJECT_NOT_FOUND
        assert cl.migrate("m", bb.StorageClass.RAM_GPU) == bb.ErrorCode.INSUFFICIENT_SPACE  # no such tier in this cluster
        assert "bb_migrations_total 2" in c.keystone.metrics_text()


def test_fault_injection_corruption_and_read_errors_fail_over_to_replica(bb):
    """BB_FAULT hooks (csrc/common/fault.h): a silently corrupted replica is caught by the per-shard digest and the
    get is served from the other copy; an I/O error on one data server does the same; a failed write cancels the put."""
    with LocalCluster("faults", n_workers=2, pool_bytes=16 << 20) as c:
        cl = c.client()
        cfg = bb.WorkerConfig(replication_factor=2, max_workers_per_copy=1, ttl_ms=0, checksum=bb.ChecksumAlgo.CRC32C)
        blob = os.urandom(300_000)
        try:
            bb.fault_arm("corrupt_write", 1, 1)  # exactly one shard write is corrupted after it lands
            assert cl.put("c1", blob, cfg) == bb.ErrorCode.OK
            bb.fault_clear()
            for _ in range(4):  # whichever replica is tried first, the answer is the intact one
                assert cl.get("c1") == blob
            assert cl.phase_summary() is not None
            assert cl.put("c1b", blob, cfg) == bb.ErrorCode.OK  # two intact replicas (c1 still has its corrupted one)
            bb.fault_arm("fail_data_read", 1, 1)
            assert cl.get("c1b") == blob  # first read errors out -> next replica
            bb.fault_arm("fail_data_write", 1, 1)
            assert cl.put("c2", blob, cfg) != bb.ErrorCode.OK
            bb.fault_clear()
            assert cl.object_exists("c2") is False  # cancelled, nothing half-written is visible
            assert cl.put("c2", blob, cfg) == bb.ErrorCode.OK and cl.get("c2") == blob
            bb.fault_arm("fail_put_complete", 1, 1)
            assert cl.put("c3", blob, cfg) != bb.ErrorCode.OK
            bb.fault_clear()
            assert cl.object_exists("c3") is False
            assert bb.fault_arm_from_spec("drop_heartbeat, delay_rpc_ms=5, corrupt_write:3") == 3
        finally:
            bb.fault_clear()


def test_trace_spans_are_recorded_and_dumped_as_chrome_trace(bb, tmp_path):
    import json

    bb.trace_clear()
    bb.trace_enable(True, 1024)
    try:
        with LocalCluster("trace", n_workers=1, pool_bytes=8 << 20) as c:
            cl = c.client()
            assert cl.put("t", b"x" * 5000, bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1)) == bb.ErrorCode.OK
            assert cl.get("t") == b"x" * 5000
        out = tmp_path / "trace.json"
        n = bb.trace_dump(str(out))
        ev = json.loads(out.read_text())["traceEvents"]
        assert n == len(ev) and n >= 2
        names = {e["name"] for e in ev}
        assert {"client.put", "client.get", "rpc.serve"} <= names and all(e["ph"] in ("X", "i") for e in ev)  # client phases and the servers' side of each RPC
        assert all(e["dur"] > 0 for e in ev if e["ph"] == "X")
    finally:
        bb.trace_enable(False)
        bb.trace_clear()


def test_read_driven_promotion_back_to_the_fast_tier(bb, tmp_path):
    """keystone.promote_after_reads: an object that keeps being read while it sits on a lower tier moves back up
    (bytes through the mover, digest re-checked), as long as the faster tier stays under its watermark."""
    kc = bb.KeystoneConfig()
    kc.promote_after_reads = 3
    kc.high_watermark = 0.9
    kc.health_check_interval_sec = 3600
    with LocalCluster("promo", n_workers=0, keystone_cfg=kc) as c:
        c.add_worker("w0", "node-0", [("dram", bb.StorageClass.RAM_CPU, 8 << 20, ""), ("nvme", bb.StorageClass.NVME, 64 << 20, str(tmp_path))])
        c.keystone.install_data_server_mover()
        cl = c.client()
        cold = bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1, ttl_ms=0, preferred_classes=[bb.StorageClass.NVME], checksum=bb.ChecksumAlgo.CRC32C)
        hot_blob, big_blob = os.urandom(1 << 20), os.urandom(12 << 20)
        assert cl.put("hot", hot_blob, cold) == bb.ErrorCode.OK
        assert cl.put("big", big_blob, cold) == bb.ErrorCode.OK
        assert cl.put("idle", os.urandom(1 << 20), cold) == bb.ErrorCode.OK
        for _ in range(2):
            assert cl.get("hot") == hot_blob
        assert c.keystone.run_promotion_once() == 0  # two reads: below the threshold
        assert cl.get("hot") == hot_blob
        for _ in range(3):
            assert cl.get("big") == big_blob  # hot too, but 12 MiB would push the 8 MiB DRAM tier over its watermark
        assert c.keystone.run_promotion_once() == 1
        tier = lambda k: cl.get_workers(k)[0].shards[0].storage_class  # noqa: E731
        assert tier("hot") == bb.StorageClass.RAM_CPU and tier("big") == bb.StorageClass.NVME and tier("idle") == bb.StorageClass.NVME
        assert cl.get("hot") == hot_blob and "bb_promotions_total 1" in c.keystone.metrics_text()


@pytest.mark.parametrize("algo_name", ["BBH64", "CRC32C"])
def test_large_objects_take_the_multi_stream_bulk_path(bb, algo_name):
    """Objects of tens of MiB cross the TCP data path as several parallel streams (gathered sends from the caller's
    buffer, in-place receives, zero-copy reads out of the pool); per-stream digests combine into the object digest the
    Keystone records, and corruption in the pool is caught on the way back."""
    algo = getattr(bb.ChecksumAlgo, algo_name)
    with LocalCluster(cluster_id=f"bulk-{algo_name}", n_workers=2, pool_bytes=256 << 20) as c:
        cl = c.client(io_parallelism=4)
        size = (40 << 20) + 12345  # not a multiple of the chunk, the stream split or the BBH64 tile
        data = os.urandom(size)
        cfg = bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1, checksum=algo)
        assert cl.put("big", data, cfg) == bb.ErrorCode.OK
        sh = cl.get_workers("big")[0].shards[0]
        want = bb.bbh64_reference(data) if algo_name == "BBH64" else bb.crc32c(data)
        assert sh.length == size and sh.checksum == want and sh.checksum_algo == algo
        assert cl.get("big") == data
        # striped over both workers + replicated: every shard is its own bulk transfer
        cfg2 = bb.WorkerConfig(replication_factor=2, max_workers_per_copy=2, checksum=algo)
        assert cl.put("big2", data, cfg2) == bb.ErrorCode.OK
        assert cl.get("big2") == data
        # flip one byte inside the pool: the verified get reports it (single copy -> CHECKSUM_MISMATCH)
        pool = [p for p in cl.keystone().get_memory_pools() if p.id == sh.pool_id][0]
        w = [w for w in c.workers if w.backend(sh.pool_id) is not None][0]
        w.backend(sh.pool_id).write(sh.location["remote_addr"] - pool.ucx_remote_addr + (33 << 20), b"\x00\x01\x02\x03")
        with pytest.raises(Exception):
            cl.get("big")


def test_worker_serves_its_own_prometheus_endpoint(bb):
    """Workers expose per-pool capacity / usage / traffic counters on /metrics (plus /healthz, /stats) when
    `http_metrics_port` is set -- the Keystone's endpoint only has the cluster-wide view."""
    with LocalCluster(cluster_id="wmetrics", n_workers=0) as c:
        wc = bb.WorkerServiceConfig()
        wc.worker_id, wc.node_id, wc.cluster_id = "wm", "node-wm", "wmetrics"
        wc.ucx_endpoint = "127.0.0.1:0"
        wc.http_metrics_port = 0  # ephemeral
        wc.storage_pools = [bb.StoragePoolConfig("ram-wm", bb.StorageClass.RAM_CPU, 32 << 20, "")]
        w = bb.WorkerService(wc, bb.CoordService(c.coord_uri))
        assert w.create_storage_pools_from_config() == bb.ErrorCode.OK and w.initialize() == bb.ErrorCode.OK and w.start() == bb.ErrorCode.OK
        c.workers.append(w)
        c.coord.store().flush_events()
        cl = c.client()
        data = os.urandom(100_000)
        assert cl.put("m", data, bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1)) == bb.ErrorCode.OK
        assert cl.get("m") == data
        status, text = bb.http_get("127.0.0.1", w.http_port, "/metrics")
        assert status == 200 and text == w.metrics_text() or "bb_pool_bytes_written_total" in text
        lines = {ln.split(" ")[0]: ln.split(" ")[1] for ln in text.splitlines() if ln and not ln.startswith("#")}
        lab = 'worker="wm",node="node-wm",pool="ram-wm",tier="RAM_CPU"'
        assert lines[f"bb_pool_capacity_bytes{{{lab}}}"] == str(32 << 20)
        assert int(lines[f"bb_pool_bytes_written_total{{{lab}}}"]) >= len(data) and int(lines[f"bb_pool_bytes_read_total{{{lab}}}"]) >= len(data)
        assert f"bb_pool_reserved_bytes{{{lab}}}" in lines and lines['bb_worker_up{worker="wm",node="node-wm"}'] == "1"
        assert bb.http_get("127.0.0.1", w.http_port, "/healthz")[0] == 200
        import json as _json
        st = _json.loads(bb.http_get("127.0.0.1", w.http_port, "/stats")[1])
        assert st["worker_id"] == "wm" and st["pools"][0]["pool_id"] == "ram-wm"


def test_admin_calls_over_rpc_workers_info_and_remove_worker(bb):
    """Reference admin surface (keystone_service.h:105-165) through the RPC client: get_workers_info lists workers with
    heartbeat age and pools; remove_worker decommissions one (works with a coordination store, where the reference
    throws): its copies are invalidated, a replicated object stays readable from the other worker."""
    with LocalCluster(cluster_id="admin", n_workers=2) as c:
        cl = c.client()
        data = os.urandom(20_000)
        assert cl.put("r2", data, bb.WorkerConfig(replication_factor=2, max_workers_per_copy=1)) == bb.ErrorCode.OK
        ws = cl.keystone().get_workers_info()
        assert sorted(w["worker_id"] for w in ws) == ["worker-0", "worker-1"]
        assert all(w["pools"] and w["heartbeat_age_ms"] >= 0 and w["node_id"].startswith("node-") for w in ws)
        assert cl.keystone().remove_worker("worker-0") == bb.ErrorCode.OK
        c.coord.store().flush_events()
        assert [w["worker_id"] for w in cl.keystone().get_workers_info()] == ["worker-1"]
        assert cl.get("r2") == data
        assert all(cp.shards[0].worker_id == "worker-1" for cp in cl.get_workers("r2"))
        assert cl.keystone().remove_worker("no-such-worker") != bb.ErrorCode.OK


@pytest.mark.parametrize("shm", [False, True])
def test_host_paths_are_exact_at_chunk_stream_and_tile_boundaries(bb, shm):
    """Sizes around every internal boundary of the host data paths (8 MiB request chunks, 4 MiB stream split, 1 MiB hash
    steps, 16 KiB BBH64 tiles, empty objects) survive put -> get bit-exactly on the TCP streams and on the shared-memory
    path, with both checksums, and the digest the Keystone records is the reference digest of the bytes."""
    MiB = 1 << 20
    sizes = [0, 1, 4095, 16384, 16385, MiB - 1, MiB + 1, 4 * MiB, 8 * MiB - 1, 8 * MiB, 8 * MiB + 1, 12 * MiB + 16384 + 7, 3 * 8 * MiB + 5]
    with LocalCluster(cluster_id=f"edge-{int(shm)}", n_workers=0) as c:
        wc = bb.WorkerServiceConfig()
        wc.worker_id, wc.node_id, wc.cluster_id, wc.ucx_endpoint = "we", "node-we", c.cluster_id, "127.0.0.1:0"
        pool = bb.StoragePoolConfig("ram-we", bb.StorageClass.RAM_CPU, 160 * MiB, "")
        pool.shared_memory = shm
        wc.storage_pools = [pool]
        w = bb.WorkerService(wc, bb.CoordService(c.coord_uri))
        assert w.create_storage_pools_from_config() == bb.ErrorCode.OK and w.initialize() == bb.ErrorCode.OK and w.start() == bb.ErrorCode.OK
        c.workers.append(w)
        c.coord.store().flush_events()
        o = bb.BlackbirdClientOptions("127.0.0.1", c.rpc.rpc_port, 30000, 3, "node-we")  # 3 streams: uneven splits
        o.enable_shm = shm
        cl = bb.BlackbirdClient(o)
        assert cl.connect() == bb.ErrorCode.OK
        blob = os.urandom(max(sizes))
        for algo in (bb.ChecksumAlgo.BBH64, bb.ChecksumAlgo.CRC32C):
            cfg = bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1, checksum=algo, ttl_ms=0)
            for n in sizes:
                key = f"e/{int(algo)}/{n}"
                data = blob[:n]
                assert cl.put(key, data, cfg) == bb.ErrorCode.OK, n
                assert cl.get(key) == data, n
                if n:
                    sh = cl.get_workers(key)[0].shards[0]
                    assert sh.checksum == (bb.bbh64_reference(data) if algo == bb.ChecksumAlgo.BBH64 else bb.crc32c_sw(data, 0)), n
                assert cl.remove(key) == bb.ErrorCode.OK
        text = cl.metrics_text()
        assert ("bb_client_shm_put_shards_total" in text) == shm


def test_list_objects_prefix_order_and_pagination(bb):
    """Listing (an extension: the reference has none): complete objects under a prefix, in key order, paginated;
    pending and removed objects do not show up."""
    with LocalCluster(cluster_id="ls", n_workers=2) as c:
        cl = c.client()
        cfg = bb.WorkerConfig(replication_factor=2, max_workers_per_copy=1)
        keys = [f"ds/train/{i:03d}" for i in range(25)] + ["ds/val/0", "other/x"]
        for k in keys:
            assert cl.put(k, os.urandom(100 + len(k)), cfg) == bb.ErrorCode.OK
        c.keystone.put_start("ds/train/pending", 10, cfg)  # never completed
        api = cl.keystone()
        got = api.list_objects("ds/train/")
        assert [g[0] for g in got] == sorted(k for k in keys if k.startswith("ds/train/"))
        assert all(g[1] == 100 + len(g[0]) and g[2] == 2 and g[3] == bb.StorageClass.RAM_CPU for g in got)
        page1 = api.list_objects("ds/", 10)
        page2 = api.list_objects("ds/", 10, page1[-1][0])
        page3 = api.list_objects("ds/", 10, page2[-1][0])
        assert [g[0] for g in page1 + page2 + page3] == sorted(k for k in keys if k.startswith("ds/")) and len(page3) == 6
        assert cl.remove("ds/val/0") == bb.ErrorCode.OK
        assert [g[0] for g in api.list_objects("ds/val")] == [] and len(api.list_objects()) == 26


def test_compact_pool_moves_high_objects_into_holes_and_frees_the_tail(bb):
    """Pool compaction (a roadmap item of the reference): after removals leave holes, a put that needs one large extent
    fails although enough bytes are free; compact_pool re-places the objects that sit highest into the holes (data moved
    by the workers, digests re-checked, placements swapped atomically) and the same put then succeeds."""
    MiB = 1 << 20
    with LocalCluster(cluster_id="compact", n_workers=1, pool_bytes=8 * MiB) as c:
        c.keystone.install_data_server_mover()
        cl = c.client()
        cfg = bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1, ttl_ms=0, checksum=bb.ChecksumAlgo.CRC32C)
        blobs = {k: os.urandom(MiB) for k in "abcdef"}
        for k, v in blobs.items():
            assert cl.put(k, v, cfg) == bb.ErrorCode.OK
        for k in "ace":  # holes at 0, 2 and 4 MiB; the free tail is 2 MiB
            assert cl.remove(k) == bb.ErrorCode.OK
        big = os.urandom(4 * MiB)
        assert cl.put("big", big, cfg) == bb.ErrorCode.INSUFFICIENT_SPACE  # 5 MiB free, largest hole 2 MiB
        api = cl.keystone()
        frag_before = [p for p in api.get_memory_pools() if p.id == "pool-0"][0]
        moved = api.compact_pool("pool-0")
        assert moved >= 2
        tops = {}
        for k in "bdf":
            sh = cl.get_workers(k)[0].shards[0]
            tops[k] = sh.location["remote_addr"] - frag_before.ucx_remote_addr + sh.length
            assert cl.get(k) == blobs[k] and sh.checksum == bb.crc32c(blobs[k])
        assert max(tops.values()) <= 3 * MiB + 4096  # the three survivors are packed at the bottom
        assert cl.put("big", big, cfg) == bb.ErrorCode.OK and cl.get("big") == big
        assert api.compact_pool("pool-0") == 0  # nothing left to gain
        with pytest.raises(bb.BlackbirdError) as e:
            api.compact_pool("no-such-pool")
        assert e.value.code == bb.ErrorCode.MEMORY_POOL_NOT_FOUND
        assert "bb_compaction_moves_total" in c.keystone.metrics_text()
        # automatic trigger: off by default, armed by compaction_fragmentation_threshold (run by the health loop)
        for k in ("big", "d"):
            assert cl.remove(k) == bb.ErrorCode.OK
        assert c.keystone.run_compaction_once() == 0


def test_health_loop_compacts_pools_above_the_fragmentation_threshold(bb):
    MiB = 1 << 20
    kc = bb.KeystoneConfig()
    kc.compaction_fragmentation_threshold = 0.3
    with LocalCluster(cluster_id="autocompact", n_workers=1, pool_bytes=8 * MiB, keystone_cfg=kc) as c:
        c.keystone.install_data_server_mover()
        cl = c.client()
        cfg = bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1, ttl_ms=0)
        blobs = {k: os.urandom(MiB) for k in "abcdef"}
        for k, v in blobs.items():
            assert cl.put(k, v, cfg) == bb.ErrorCode.OK
        for k in "ace":
            assert cl.remove(k) == bb.ErrorCode.OK
        pool = lambda: [p for p in cl.keystone().get_memory_pools() if p.id == "pool-0"][0]  # noqa: E731
        assert c.keystone.run_compaction_once() >= 2  # what the health loop does every health_check_interval_sec
        assert all(cl.get(k) == blobs[k] for k in "bdf")
        assert cl.put("big", os.urandom(4 * MiB), cfg) == bb.ErrorCode.OK and pool().used >= 7 * MiB
        assert c.keystone.run_compaction_once() == 0


def test_readers_survive_concurrent_compaction_and_migration(bb):
    """Gets that lose a race with the Keystone moving an object (compaction, explicit migration) re-read the placements
    and succeed: no reader ever sees an error or wrong bytes while objects are being shuffled underneath."""
    import random
    import threading
    import time

    MiB = 1 << 20
    with LocalCluster(cluster_id="shuffle", n_workers=1, pool_bytes=24 * MiB) as c:
        c.keystone.install_data_server_mover()
        c.add_worker("worker-disk", "node-0", [("disk-0", bb.StorageClass.HDD, 64 * MiB, "/tmp")])
        cl = c.client()
        cfg = bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1, ttl_ms=0, preferred_classes=[bb.StorageClass.RAM_CPU])
        blobs = {f"o{i}": os.urandom(MiB // 2 + 1000 * i) for i in range(14)}
        for k, v in blobs.items():
            assert cl.put(k, v, cfg) == bb.ErrorCode.OK
        stop = threading.Event()
        errors, reads = [], [0]

        def reader(seed):
            rc = c.client()
            rng = random.Random(seed)
            while not stop.is_set():
                k = rng.choice(list(blobs))
                try:
                    if rc.get(k) != blobs[k]:
                        errors.append((k, "wrong bytes"))
                except Exception as e:  # noqa: BLE001
                    errors.append((k, repr(e)))
                reads[0] += 1

        ts = [threading.Thread(target=reader, args=(s,)) for s in range(3)]
        [t.start() for t in ts]
        api = cl.keystone()
        rng = random.Random(7)
        moves = 0
        t_end = time.time() + 2.0
        while time.time() < t_end:
            k = rng.choice(list(blobs))
            assert cl.remove(k) == bb.ErrorCode.OK  # open a hole ...
            moves += api.compact_pool("pool-0", 4)   # ... let compaction fill it ...
            assert cl.put(k, blobs[k], cfg) == bb.ErrorCode.OK
            k2 = rng.choice([x for x in blobs if x != k])
            tier = cl.get_workers(k2)[0].shards[0].storage_class  # ... and bounce another object between tiers
            assert cl.migrate(k2, bb.StorageClass.HDD if tier == bb.StorageClass.RAM_CPU else bb.StorageClass.RAM_CPU) == bb.ErrorCode.OK
        stop.set()
        [t.join() for t in ts]
        # a reader may legitimately see OBJECT_NOT_FOUND / NOT_READY for the key that is being removed and re-put
        hard = [e for e in errors if "OBJECT_NOT_FOUND" not in e[1] and "OBJECT_NOT_READY" not in e[1]]
        assert not hard, hard[:5]
        assert reads[0] > 50 and moves > 0


def test_put_straddling_a_keystone_failover_is_restarted(bb):
    """The leader dies between a client's put_start and its put_complete.  The pending object was never in the metadata
    log, so the new leader answers OBJECT_NOT_FOUND to the put_complete -- the client (which knows both keystones)
    notices that it failed over in the middle of the put and runs it again instead of returning that error."""
    import threading
    import time

    kc = bb.KeystoneConfig()
    kc.enable_ha = True
    kc.service_id = "ks-a"
    kc.service_registration_ttl_sec = 2
    kc.service_refresh_interval_sec = 1
    with LocalCluster(cluster_id="ha-put", n_workers=1, keystone_cfg=kc) as c:
        kb = bb.KeystoneConfig()
        kb.enable_ha, kb.service_id, kb.service_registration_ttl_sec, kb.service_refresh_interval_sec = True, "ks-b", 2, 1
        kb.cluster_id, kb.listen_address, kb.http_metrics_port = "ha-put", "127.0.0.1:0", "0"
        b = bb.KeystoneService(kb, bb.CoordService(c.coord_uri))
        assert b.initialize() == bb.ErrorCode.OK and b.start() == bb.ErrorCode.OK
        rb = bb.RpcService(b, kb)
        assert rb.start() == bb.ErrorCode.OK
        try:
            assert c.keystone.is_leader() and not b.is_leader()
            c.coord.store().flush_events()
            opts = bb.BlackbirdClientOptions()
            opts.keystone_endpoints = [f"127.0.0.1:{c.rpc.rpc_port}", f"127.0.0.1:{rb.rpc_port}"]
            cl = bb.BlackbirdClient(opts)
            assert cl.connect() == bb.ErrorCode.OK
            cl.keystone().set_failover_budget_ms(20000)
            data = os.urandom(300_000)
            wc = bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1)
            assert cl.put("warm", data, wc) == bb.ErrorCode.OK
            out = []
            bb.fault_arm("delay_rpc_ms", 400)  # every RPC takes 0.4 s: put_start | data write | put_complete
            t = threading.Thread(target=lambda: out.append(cl.put("straddler", data, wc)))
            t.start()
            time.sleep(0.6)  # put_start has been answered by ks-a, the shard is on its way to the worker
            c.rpc.stop()
            c.keystone.stop()
            t.join(timeout=40)
            bb.fault_clear()
            assert not t.is_alive() and out == [bb.ErrorCode.OK], out
            assert b.is_leader() and cl.keystone().failovers() >= 1
            assert cl.get("straddler") == data and cl.get("warm") == data  # "warm" came back through the metadata log
            assert "put_restarted_after_failover_total 1" in cl.metrics_text()
        finally:
            bb.fault_clear()
            rb.stop()
            b.stop()


def test_xxh3_digest_on_the_host_path_put_get_and_corruption(bb):
    """ChecksumAlgo.XXH3 through the TCP data path: parallel streams hash their tile ranges and the sums add up to the
    digest the GPU kernels produce for the same bytes (bb.xxh3t64 is the shared model)."""
    import os

    from blackbird_b200.parallel import LocalCluster

    with LocalCluster("xxh3-host", n_workers=2, pool_bytes=32 << 20) as c:
        cl = c.client(io_parallelism=4)
        wc = bb.WorkerConfig(replication_factor=2, max_workers_per_copy=1, ttl_ms=0, checksum=bb.ChecksumAlgo.XXH3)
        blob = os.urandom((9 << 20) + 12345)
        assert cl.put("x", blob, wc) == bb.ErrorCode.OK
        copies = cl.get_workers("x")
        assert all(cp.shards[0].checksum == bb.xxh3t64(blob) and cp.shards[0].checksum_algo == bb.ChecksumAlgo.XXH3 for cp in copies)
        assert cl.get("x") == blob
        sh = copies[0].shards[0]
        w = next(w for i, w in enumerate(c.workers) if f"pool-{i}" == sh.pool_id)
        w.backend(sh.pool_id).write(sh.location["remote_addr"] - w.backend(sh.pool_id).get_base_address() + 5000, b"\x00\x01\x02\x03")
        assert cl.get("x") == blob  # digest mismatch on replica 0 -> served from replica 1


def test_drain_worker_moves_everything_off_before_the_worker_leaves(bb, tmp_path):
    """`drain_worker` (bb-cli drain-worker ID): the graceful form of remove-worker.  The worker's pools stop taking placements,
    every object with a shard there is re-placed on the others while the old copies keep serving, nothing is ever degraded or
    lost, and the worker is removed at the end."""
    with LocalCluster("drain", n_workers=0) as c:
        for i in range(3):
            c.add_worker(f"w{i}", f"n{i}", [(f"dram{i}", bb.StorageClass.RAM_CPU, 16 << 20, ""), (f"nvme{i}", bb.StorageClass.NVME, 16 << 20, str(tmp_path / f"d{i}"))])
        c.keystone.install_data_server_mover()
        cl = c.client()
        blobs = {}
        for i in range(12):
            cfg = bb.WorkerConfig(replication_factor=2 if i % 2 else 1, max_workers_per_copy=1, ttl_ms=0,
                                  preferred_classes=[bb.StorageClass.RAM_CPU if i % 3 else bb.StorageClass.NVME])
            blobs[f"d/{i}"] = os.urandom(200_000 + i)
            assert cl.put(f"d/{i}", blobs[f"d/{i}"], cfg) == bb.ErrorCode.OK
        on_w0 = [k for k in blobs if any(s.worker_id == "w0" for cp in cl.get_workers(k) for s in cp.shards)]
        assert on_w0, "the test needs objects on the worker it drains"
        copies_before = {k: len(cl.get_workers(k)) for k in blobs}
        elsewhere = {k: [(s.pool_id, s.offset) for cp in cl.get_workers(k) for s in cp.shards if s.worker_id != "w0"] for k in blobs}
        moved = c.keystone.drain_worker("w0")
        assert moved == len(on_w0)
        for k in blobs:  # only what touched w0 moved: a replica on another worker is exactly where it was
            now = [(s.pool_id, s.offset) for cp in cl.get_workers(k) for s in cp.shards]
            assert all(x in now for x in elsewhere[k]), (k, elsewhere[k], now)
            assert len({s.worker_id for cp in cl.get_workers(k) for s in cp.shards}) == copies_before[k]  # one replica per worker still
        assert all(w["worker_id"] != "w0" for w in cl.keystone().get_workers_info())
        for k, v in blobs.items():
            placed = cl.get_workers(k)
            assert len(placed) == copies_before[k]  # same redundancy as before: nothing was degraded on the way
            assert all(s.worker_id != "w0" for cp in placed for s in cp.shards)
            assert cl.get(k) == v
        # every copy, not just the one a read happens to pick (a padded O_DIRECT write used to wipe the head of the object
        # stored behind the one being moved; the read path hid it by failing over to the other replica)
        rep = c.keystone.scrub()
        assert rep["objects"] == len(blobs) and rep["corrupt"] == 0 and rep["unreachable"] == 0
        text = c.keystone.metrics_text()
        assert f"bb_drain_moves_total {len(on_w0)}" in text and ("bb_objects_lost_total 0" in text or "bb_objects_lost_total" not in text)
        # new objects avoid nothing now; a second drain of a worker that is gone is an error, not a crash
        assert cl.put("after", b"x" * 1000, bb.WorkerConfig(replication_factor=2, max_workers_per_copy=1)) == bb.ErrorCode.OK
        with pytest.raises(bb.BlackbirdError) as e:
            c.keystone.drain_worker("w0")
        assert e.value.code == bb.ErrorCode.INVALID_WORKER


def test_drain_worker_without_room_elsewhere_keeps_the_worker_and_its_objects(bb):
    """No space on the other workers: nothing is lost, the objects stay where they are, the call says INSUFFICIENT_SPACE and
    the worker stays registered (draining: it takes no new placements until the drain is repeated or it is removed)."""
    with LocalCluster("drain2", n_workers=0) as c:
        c.add_worker("big", "n0", [("dram-big", bb.StorageClass.RAM_CPU, 8 << 20, "")])
        c.add_worker("tiny", "n1", [("dram-tiny", bb.StorageClass.RAM_CPU, 1 << 20, "")])
        c.keystone.install_data_server_mover()
        cl = c.client()
        cfg = bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1, ttl_ms=0, preferred_node="n0")
        blobs = {f"k{i}": os.urandom(900_000) for i in range(4)}
        for k, v in blobs.items():
            assert cl.put(k, v, cfg) == bb.ErrorCode.OK
        with pytest.raises(bb.BlackbirdError) as e:
            c.keystone.drain_worker("big")
        assert e.value.code == bb.ErrorCode.INSUFFICIENT_SPACE
        assert any(w["worker_id"] == "big" for w in cl.keystone().get_workers_info())
        for k, v in blobs.items():
            assert cl.get(k) == v
        # draining: new objects go elsewhere (or nowhere), never onto the worker that is leaving
        r = cl.put("new-small", b"y" * 1000, bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1))
        if r == bb.ErrorCode.OK:
            assert all(s.worker_id != "big" for cp in cl.get_workers("new-small") for s in cp.shards)


def _rot(cluster, shard, at=1000, n=64):
    """Silent corruption of a stored shard: bytes change inside the pool, nobody is told."""
    w = next(w for w in cluster.workers if w.data_endpoint() == f"{shard.endpoint.ip}:{shard.endpoint.port}")
    b = w.backend(shard.pool_id)
    off = shard.offset - (b.get_base_address() if shard.location["kind"] == "memory" else 0)
    old = b.read(off + at, n)
    assert int(b.write(off + at, bytes(x ^ 0x5A for x in old))) == 0


@pytest.mark.parametrize("tier", ["RAM_CPU", "NVME"])
def test_scrub_finds_a_rotted_copy_and_replaces_it_from_a_healthy_one(bb, tmp_path, tier):
    """Scrub (the reference never re-reads what it stored): the workers hash every copy where it lies; the copy that no longer
    matches its digest is replaced by a fresh one made from a replica that does, its extents go back to the allocator, and the
    next scrub finds nothing.  Without it the rot waits for a read -- or for the day the healthy replica's worker dies."""
    sc = getattr(bb.StorageClass, tier)
    with LocalCluster("scrub", n_workers=0) as c:
        for i in range(3):
            c.add_worker(f"w{i}", f"n{i}", [(f"p{i}", sc, 16 << 20, str(tmp_path / f"d{i}") if tier == "NVME" else "")])
        c.keystone.install_data_server_mover()
        cl = c.client()
        cfg = bb.WorkerConfig(replication_factor=2, max_workers_per_copy=1, ttl_ms=0)
        blobs = {f"s/{i}": os.urandom(300_000 + 17 * i) for i in range(6)}
        for k, v in blobs.items():
            assert cl.put(k, v, cfg) == bb.ErrorCode.OK
        clean = c.keystone.scrub()
        assert clean == {"objects": 6, "copies": 12, "corrupt": 0, "healed": 0, "unrecoverable": 0, "unreachable": 0}
        victim = cl.get_workers("s/2")[1]
        survivor_pool = cl.get_workers("s/2")[0].shards[0].pool_id
        _rot(c, victim.shards[0])
        rep = cl.keystone().scrub("s/")  # the same call over RPC-shaped API (bb-cli scrub)
        assert rep["corrupt"] == 1 and rep["healed"] == 1 and rep["unrecoverable"] == 0 and rep["objects"] == 6
        after = cl.get_workers("s/2")
        assert len(after) == 2 and after[0].shards[0].pool_id == survivor_pool
        fresh = after[1].shards[0]
        assert fresh.pool_id != survivor_pool  # still one replica per pool
        assert (fresh.pool_id, fresh.offset) != (victim.shards[0].pool_id, victim.shards[0].offset)  # new extents, not a patch in place
        assert c.keystone.scrub() == clean  # every copy of every object matches again
        for k, v in blobs.items():
            assert cl.get(k) == v
        text = c.keystone.metrics_text()
        assert "bb_scrub_corrupt_copies_total 1" in text and "bb_scrub_healed_total 1" in text
        # the bad extents went back: removing everything leaves the pools empty
        for k in blobs:
            assert cl.remove(k) == bb.ErrorCode.OK
        assert cl.cluster_stats().used_capacity == 0


def test_scrub_reports_an_object_with_no_healthy_copy_left(bb):
    """One replica, rotted: there is nothing to heal from.  The object stays listed, scrub says so (bb-cli exits 2), the metric
    counts it, and a read fails its digest check instead of returning the wrong bytes."""
    with LocalCluster("scrub1", n_workers=2) as c:
        c.keystone.install_data_server_mover()
        cl = c.client()
        blob = os.urandom(100_000)
        assert cl.put("only", blob, bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1)) == bb.ErrorCode.OK
        assert cl.put("fine", blob, bb.WorkerConfig(replication_factor=2, max_workers_per_copy=1)) == bb.ErrorCode.OK
        _rot(c, cl.get_workers("only")[0].shards[0], at=0, n=8)
        rep = c.keystone.scrub()
        assert rep["objects"] == 2 and rep["corrupt"] == 1 and rep["healed"] == 0 and rep["unrecoverable"] == 1
        assert cl.object_exists("only") and "bb_scrub_unrecoverable_total 1" in c.keystone.metrics_text()
        with pytest.raises(bb.BlackbirdError) as e:
            cl.get("only")
        assert e.value.code == bb.ErrorCode.CHECKSUM_MISMATCH
        assert c.keystone.scrub("fine", 1)["objects"] == 1  # prefix + object budget


def test_repair_uses_a_copy_that_verifies_when_the_first_one_rotted(bb):
    """Re-replication after a worker death reads a surviving copy; if that copy fails its digest on the way the next one is
    used (the first was the only candidate before: a rotted copy 0 blocked the repair for good)."""
    with LocalCluster("rep", n_workers=4) as c:
        c.keystone.install_data_server_mover()
        cl = c.client()
        blob = os.urandom(200_000)
        assert cl.put("r3", blob, bb.WorkerConfig(replication_factor=3, max_workers_per_copy=1, ttl_ms=0)) == bb.ErrorCode.OK
        copies = cl.get_workers("r3")
        _rot(c, copies[0].shards[0])
        assert c.keystone.remove_worker(copies[2].shards[0].worker_id) == bb.ErrorCode.OK  # degraded: 2 of 3 copies left
        assert len(cl.get_workers("r3")) == 2
        assert c.keystone.run_repair_once() == 1
        assert len(cl.get_workers("r3")) == 3
        rep = c.keystone.scrub()  # ... and scrub then replaces the rotted one as well
        assert rep["corrupt"] == 1 and rep["healed"] == 1
        assert c.keystone.scrub()["corrupt"] == 0 and cl.get("r3") == blob


def test_scrub_runs_next_to_writers_removers_and_rot(bb):
    """Scrub while objects are being replaced and removed and copies keep rotting: it never swaps a copy of an object that was
    replaced in the meantime, readers never see wrong bytes, and when everything is removed the pools are empty again (no extent
    of a swapped-out copy is leaked or freed twice)."""
    import random
    import threading
    import time

    with LocalCluster("scrubrace", n_workers=3, pool_bytes=32 << 20) as c:
        c.keystone.install_data_server_mover()
        cl = c.client()
        cfg = bb.WorkerConfig(replication_factor=2, max_workers_per_copy=1, ttl_ms=0)
        blobs = {f"k{i}": os.urandom(150_000 + 333 * i) for i in range(10)}
        for k, v in blobs.items():
            assert cl.put(k, v, cfg) == bb.ErrorCode.OK
        stop = threading.Event()
        errors, totals = [], {"corrupt": 0, "healed": 0, "rounds": 0}
        lock = threading.Lock()

        def scrubber():
            while not stop.is_set():
                rep = c.keystone.scrub()
                totals["corrupt"] += rep["corrupt"]
                totals["healed"] += rep["healed"]
                totals["rounds"] += 1

        def churn(seed):
            rc, rng = c.client(), random.Random(seed)
            while not stop.is_set():
                k = rng.choice(list(blobs))
                with lock:  # one writer per key at a time; scrub is the one running unsynchronised
                    if rng.random() < 0.5:
                        new = os.urandom(len(blobs[k]))
                        rc.remove(k)
                        if rc.put(k, new, cfg) != bb.ErrorCode.OK:
                            errors.append((k, "put failed"))
                        blobs[k] = new
                    else:
                        try:
                            if rc.get(k) != blobs[k]:
                                errors.append((k, "wrong bytes"))
                        except Exception as e:  # noqa: BLE001
                            errors.append((k, repr(e)))

        def rotter():
            rng = random.Random(3)
            while not stop.is_set():
                k = rng.choice(list(blobs))
                with lock:
                    try:
                        copies = cl.get_workers(k)
                        _rot(c, copies[-1].shards[0], at=rng.randrange(0, 1000), n=16)  # copy 0 stays clean: always one to heal from
                    except bb.BlackbirdError:
                        pass
                time.sleep(0.02)

        ts = [threading.Thread(target=scrubber), threading.Thread(target=rotter)] + [threading.Thread(target=churn, args=(s,)) for s in range(2)]
        [t.start() for t in ts]
        time.sleep(2.5)
        stop.set()
        [t.join() for t in ts]
        assert not errors, errors[:5]
        assert totals["rounds"] >= 2 and totals["healed"] >= 1, totals
        last = c.keystone.scrub()  # settles what the rotter did after the scrubber's last round
        assert last["unrecoverable"] == 0 and c.keystone.scrub()["corrupt"] == 0
        for k, v in blobs.items():
            assert cl.get(k) == v
        for k in blobs:
            assert cl.remove(k) == bb.ErrorCode.OK
        assert cl.cluster_stats().used_capacity == 0


def test_background_scrub_heals_without_being_asked(bb):
    """`keystone.scrub_objects_per_round`: the health loop walks the objects a slice at a time and replaces what rotted."""
    import time

    cfg = bb.KeystoneConfig()
    cfg.health_check_interval_sec = 1
    cfg.scrub_objects_per_round = 4  # 10 objects: a full pass takes a few rounds, resuming where the last one stopped
    with LocalCluster("bgscrub", n_workers=3, keystone_cfg=cfg) as c:
        c.keystone.install_data_server_mover()
        cl = c.client()
        blobs = {f"b{i}": os.urandom(50_000 + i) for i in range(10)}
        for k, v in blobs.items():
            assert cl.put(k, v, bb.WorkerConfig(replication_factor=2, max_workers_per_copy=1, ttl_ms=0)) == bb.ErrorCode.OK
        for k in ("b3", "b8"):
            _rot(c, cl.get_workers(k)[1].shards[0])
        deadline = time.time() + 20
        while time.time() < deadline and "bb_scrub_healed_total 2" not in c.keystone.metrics_text():
            time.sleep(0.2)
        text = c.keystone.metrics_text()
        assert "bb_scrub_healed_total 2" in text and "bb_scrub_corrupt_copies_total 2" in text, [l for l in text.splitlines() if "scrub" in l]
        assert c.keystone.scrub()["corrupt"] == 0
        for k, v in blobs.items():
            assert cl.get(k) == v
