"""Reservation protocol between the Keystone and the workers (reference storage_backend.h:46-126: reserve_shard ->
commit_shard | abort_shard, free_shard -- implemented there, called by no service; VERDICT r1 A10).

put_start -> the Keystone reserves every shard AT ITS WORKER (token with an expiry) -> the client writes -> put_complete
commits the tokens -> remove frees the committed shards.  A writer that vanishes is cleaned up by the worker: its tokens
expire, the backend takes the ranges back, the worker reports through the coordination store and the Keystone drops the
PENDING object -- with the Keystone's own GC switched off."""
import os
import time

import pytest

from blackbird_b200.parallel import LocalCluster


def wait_for(pred, timeout=8.0, step=0.02):
    deadline = time.time() + timeout
    while time.time() < deadline:
        if pred():
            return True
        time.sleep(step)
    return pred()


@pytest.fixture
def rcluster(bb):
    cfg = bb.KeystoneConfig()
    cfg.enable_gc = False            # nothing on the Keystone side may clean up for the worker
    cfg.gc_interval_sec = 3600
    cfg.health_check_interval_sec = 3600
    cfg.enable_reservations = True
    cfg.reservation_ttl_ms = 400
    c = LocalCluster("resv", n_workers=2, pool_bytes=8 << 20, keystone_cfg=cfg)
    c.keystone.install_reservation_hooks()
    yield c
    c.stop()


def pool_stats(c):
    return {f"worker-{i}": w.backend(f"pool-{i}").get_stats() for i, w in enumerate(c.workers)}


def test_put_reserves_commits_and_remove_frees_at_the_workers(bb, rcluster):
    c = rcluster
    cl = c.client()
    wc = bb.WorkerConfig(replication_factor=2, max_workers_per_copy=1, ttl_ms=0)
    blob = os.urandom(100_000)
    placed = c.keystone.put_start("k-manual", len(blob), wc)
    st = pool_stats(c)
    assert all(s.num_reservations == 1 and s.num_committed_shards == 0 for s in st.values())  # one replica per worker, reserved
    assert all(s.used_capacity >= len(blob) for s in st.values())  # worker-side accounting sees the placement
    assert c.keystone.put_complete("k-manual") == bb.ErrorCode.OK
    st = pool_stats(c)
    assert all(s.num_reservations == 0 and s.num_committed_shards == 1 for s in st.values())
    # the full client path (put = put_start + data + put_complete) goes through the same protocol
    assert cl.put("k-client", blob, wc) == bb.ErrorCode.OK and cl.get("k-client") == blob
    assert all(s.num_committed_shards == 2 for s in pool_stats(c).values())
    # remove -> free_shard at the workers; cancel of a PENDING put -> abort
    assert cl.remove("k-client") == bb.ErrorCode.OK and cl.remove("k-manual") == bb.ErrorCode.OK
    c.keystone.put_start("k-cancel", 4096, wc)
    assert all(s.num_reservations == 1 for s in pool_stats(c).values())
    assert c.keystone.put_cancel("k-cancel") == bb.ErrorCode.OK
    st = pool_stats(c)
    assert all(s.num_reservations == 0 and s.num_committed_shards == 0 and s.used_capacity == 0 for s in st.values())
    assert c.keystone.get_cluster_stats().used_capacity == 0  # Keystone ledger and worker stats agree
    assert placed[0].shards[0].pool_id != placed[1].shards[0].pool_id
    text = c.keystone.metrics_text()
    assert "bb_reservations_total 3" in text


def test_crashed_writer_is_reclaimed_by_token_expiry_without_keystone_gc(bb, rcluster):
    c = rcluster
    wc = bb.WorkerConfig(replication_factor=1, max_workers_per_copy=2, ttl_ms=0, min_shard_size=4096)  # striped over both workers
    c.keystone.put_start("orphan", 64 << 10, wc)  # ... and the writer is never heard of again
    assert c.keystone.get_cluster_stats().pending_objects == 1
    assert sum(s.num_reservations for s in pool_stats(c).values()) == 2
    # worker 0 sweeps (allocation_poll_interval_ms drives this in the background; here explicitly, after the TTL)
    time.sleep(0.5)
    c.workers[0].reap_reservations()  # (the background sweep may have beaten us to it)
    # the worker's report reaches the Keystone through the coordination store: the PENDING object and its ledger entry go,
    # and the object's OTHER shard, reserved at worker 1, is aborted there
    assert wait_for(lambda: c.keystone.get_cluster_stats().pending_objects == 0)
    assert wait_for(lambda: sum(s.num_reservations for s in pool_stats(c).values()) == 0)
    assert c.keystone.get_cluster_stats().used_capacity == 0 and all(s.used_capacity == 0 for s in pool_stats(c).values())
    # the watcher thread that handled the report counts it after dropping the object, so the counter may trail the state
    assert wait_for(lambda: "bb_reservation_expired_total 1" in c.keystone.metrics_text())
    # the key is free again
    assert c.keystone.put_start("orphan", 1024, bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1))
    # a put_complete that arrives after the token ran out fails: the worker has already given the range away
    time.sleep(0.5)
    for w in c.workers:
        w.reap_reservations()
    assert c.keystone.put_complete("orphan") != bb.ErrorCode.OK


def test_reservations_are_off_by_default_and_the_background_sweep_runs(bb):
    with LocalCluster("resv-off", n_workers=1, pool_bytes=4 << 20) as c:
        c.keystone.install_reservation_hooks()
        c.keystone.put_start("k", 4096, bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1))
        assert c.workers[0].backend("pool-0").get_stats().num_reservations == 0  # enable_reservations is false
    cfg = bb.KeystoneConfig()
    cfg.enable_gc = False
    cfg.enable_reservations = True
    cfg.reservation_ttl_ms = 200
    with LocalCluster("resv-bg", n_workers=1, pool_bytes=4 << 20, keystone_cfg=cfg) as c:
        c.keystone.install_reservation_hooks()
        c.keystone.put_start("k", 4096, bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1))
        # default allocation_poll_interval_ms = 1000: the reaper thread finds the expired token on its own
        assert wait_for(lambda: c.keystone.get_cluster_stats().pending_objects == 0, timeout=6)


def test_run_placed_batches_go_through_the_reservation_protocol(bb, rcluster):
    """A uniform batch is placed as a run (one allocator call per chunk); every object still gets its own reservation token at
    the worker, commits and cancels still resolve them one by one, and the Keystone ledger and the workers' stats agree."""
    c = rcluster
    wc = bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1, ttl_ms=0)
    keys = [f"rb/{i:02d}" for i in range(24)]
    res = c.keystone.batch_put_start(keys, [16384] * 24, wc)
    assert all(r[0] == bb.ErrorCode.OK for r in res)
    per_pool = {}
    for r in res:
        per_pool[r[1][0].shards[0].pool_id] = per_pool.get(r[1][0].shards[0].pool_id, 0) + 1
    st = pool_stats(c)
    assert sum(s.num_reservations for s in st.values()) == 24 and sum(s.num_committed_shards for s in st.values()) == 0
    assert sorted(per_pool.values()) == [12, 12]  # the run was dealt out over the two equal pools
    assert set(c.keystone.batch_put_complete(keys[:16])) == {bb.ErrorCode.OK}
    assert set(c.keystone.batch_put_cancel(keys[16:])) == {bb.ErrorCode.OK}
    st = pool_stats(c)
    assert sum(s.num_reservations for s in st.values()) == 0 and sum(s.num_committed_shards for s in st.values()) == 16
    assert sum(s.used_capacity for s in st.values()) == 16 * 16384 == c.keystone.get_cluster_stats().used_capacity
    assert set(c.keystone.batch_remove_object(keys[:16])) == {bb.ErrorCode.OK}
    assert sum(s.used_capacity for s in pool_stats(c).values()) == 0 and c.keystone.get_cluster_stats().used_capacity == 0
