"""Segmented device objects (batch_put_device_gather / batch_get_device_scatter) on CPU: a HostLoopbackTransport stands in
for the GPU fabric ("device pointers" are numpy buffers), so the client logic around segment lists -- validation per
object, slicing per shard (striping, replicas), fail-over, host-staged tiers, chunking by segment count -- and the
contract that a gathered object is byte- and digest-identical to a contiguous put of the concatenation run in the CPU
suite."""
import os

import numpy as np
import pytest

from blackbird_b200.parallel import LocalCluster

MiB = 1 << 20
GUARD = 0xAB
ALGOS = ["XXH3", "CRC32C", "BBH64", "NONE"]


def make_client(bb, c, reach_disk=False):
    cl = c.client(node_id="node-0")
    io = c.client(node_id="node-0")
    bb.attach_loopback_transport(cl, io, reach_disk)
    return cl


class Layout:
    """Segments of the given lengths placed in one buffer in a shuffled order, 16-byte aligned, with guard bytes between
    them.  `segs` is the (S, 2) uint64 table in object order."""

    def __init__(self, lens, rng, fill_random=True):
        lens = [int(x) for x in lens]
        slot = [(x + 15) // 16 * 16 + 32 for x in lens]
        total = sum(slot) + 64
        raw = np.full(total + 16, GUARD, dtype=np.uint8)
        off = (-raw.ctypes.data) % 16
        self.buf = raw[off:off + total]
        self._raw = raw
        order = rng.permutation(len(lens))
        pos, starts = 32, [0] * len(lens)
        for k in order:
            starts[k] = pos
            pos += slot[k]
        self.starts, self.lens = starts, lens
        self.mask = np.zeros(total, dtype=bool)
        for s, n in zip(starts, lens):
            self.mask[s:s + n] = True
            if fill_random:
                self.buf[s:s + n] = np.frombuffer(os.urandom(n), dtype=np.uint8)
        base = self.buf.ctypes.data
        self.segs = np.array([[base + s, n] for s, n in zip(starts, lens)], dtype=np.uint64).reshape(-1, 2)

    def concat(self, first=0, count=None):
        count = len(self.lens) - first if count is None else count
        return b"".join(self.buf[self.starts[k]:self.starts[k] + self.lens[k]].tobytes() for k in range(first, first + count))

    def guards_intact(self):
        return bool(np.all(self.buf[~self.mask] == GUARD))


def split(total, rng, max_seg=64 * 1024):
    """Random split of `total` bytes: multiples of 16, the last piece takes the remainder (any length)."""
    out, left = [], total
    while left > 0:
        n = int(rng.integers(1, max_seg // 16 + 1)) * 16
        if n >= left:
            n = left
        out.append(n)
        left -= n
    return out


def cfg_for(bb, algo, **kw):
    base = dict(replication_factor=1, max_workers_per_copy=1, ttl_ms=0, preferred_classes=[bb.StorageClass.RAM_CPU])
    base.update(kw)
    return bb.WorkerConfig(checksum=getattr(bb.ChecksumAlgo, algo), **base)


def objects(rng, n):
    """Per object a list of segment lengths: small, 4 KiB, large, odd tail, single segment."""
    shapes = [[16] * 40 + [7], [4096] * 9, split(300_000, rng), [48, 4096 * 5 + 16, 32, 1000], [12345], split(200_000, rng, 1024) ]
    return [shapes[i % len(shapes)] for i in range(n)]


@pytest.mark.parametrize("algo", ALGOS)
def test_gather_put_scatter_get_round_trip_and_guards(bb, algo):
    rng = np.random.default_rng(1)
    with LocalCluster(cluster_id=f"seg-rt-{algo}", n_workers=2, pool_bytes=64 * MiB) as c:
        cl = make_client(bb, c)
        objs = objects(rng, 7)
        src = Layout([x for o in objs for x in o], rng)
        counts = [len(o) for o in objs]
        keys = [f"rt/{i}" for i in range(len(objs))]
        assert cl.batch_put_device_gather(keys, src.segs, counts, cfg_for(bb, algo), 0) == [bb.ErrorCode.OK] * len(keys)
        # read back into a different split of the same totals, in a different place
        totals = [sum(o) for o in objs]
        dst_objs = [split(t, rng, 8192) for t in totals]
        dst = Layout([x for o in dst_objs for x in o], rng, fill_random=False)
        dcounts = [len(o) for o in dst_objs]
        assert cl.batch_get_device_scatter(keys, dst.segs, dcounts, 0) == [bb.ErrorCode.OK] * len(keys)
        s = d = 0
        for i in range(len(objs)):
            assert dst.concat(d, dcounts[i]) == src.concat(s, counts[i])
            s, d = s + counts[i], d + dcounts[i]
        assert dst.guards_intact() and src.guards_intact()


@pytest.mark.parametrize("algo", ALGOS)
def test_gathered_put_stores_the_digests_of_the_concatenation(bb, algo):
    rng = np.random.default_rng(2)
    with LocalCluster(cluster_id=f"seg-eq-{algo}", n_workers=2, pool_bytes=64 * MiB) as c:
        cl = make_client(bb, c)
        objs = objects(rng, 6)
        src = Layout([x for o in objs for x in o], rng)
        counts = [len(o) for o in objs]
        cfg = cfg_for(bb, algo)
        keys = [f"g/{i}" for i in range(len(objs))]
        assert cl.batch_put_device_gather(keys, src.segs, counts, cfg, 0) == [bb.ErrorCode.OK] * len(keys)
        first = 0
        for i, k in enumerate(keys):
            blob = np.frombuffer(src.concat(first, counts[i]), dtype=np.uint8).copy()
            first += counts[i]
            assert cl.batch_put_device([f"c/{i}"], [blob.ctypes.data], [blob.size], cfg, 0) == [bb.ErrorCode.OK]
            gs = [sh.checksum for cp in cl.get_workers(k) for sh in cp.shards]
            cs = [sh.checksum for cp in cl.get_workers(f"c/{i}") for sh in cp.shards]
            assert gs == cs
            if algo == "BBH64":
                assert gs == [bb.bbh64_reference(blob)]
            elif algo == "CRC32C":
                assert gs == [bb.crc32c(blob)]


def test_gathered_and_contiguous_objects_read_back_either_way(bb):
    rng = np.random.default_rng(3)
    with LocalCluster(cluster_id="seg-interop", n_workers=2, pool_bytes=64 * MiB) as c:
        cl = make_client(bb, c)
        lens = [4096] * 5 + [16 * 100, 333]
        src = Layout(lens, rng)
        cfg = cfg_for(bb, "BBH64")
        assert cl.batch_put_device_gather(["gi"], src.segs, [len(lens)], cfg, 0) == [bb.ErrorCode.OK]
        want = src.concat()
        out = np.zeros(len(want), dtype=np.uint8)
        ecs, sizes = cl.batch_get_device(["gi"], [out.ctypes.data], [out.size], 0)
        assert ecs == [bb.ErrorCode.OK] and sizes == [len(want)] and out.tobytes() == want
        assert c.client().get("gi") == want
        # contiguous put, scattered get
        blob = np.frombuffer(os.urandom(70_000), dtype=np.uint8).copy()
        assert cl.batch_put_device(["ci"], [blob.ctypes.data], [blob.size], cfg, 0) == [bb.ErrorCode.OK]
        dst = Layout(split(blob.size, rng, 4096), rng, fill_random=False)
        assert cl.batch_get_device_scatter(["ci"], dst.segs, [len(dst.lens)], 0) == [bb.ErrorCode.OK]
        assert dst.concat() == blob.tobytes() and dst.guards_intact()


@pytest.mark.parametrize("algo", ["CRC32C", "BBH64"])
def test_striped_replicated_gather_and_scatter_fail_over(bb, algo):
    rng = np.random.default_rng(4)
    with LocalCluster(cluster_id=f"seg-stripe-{algo}", n_workers=4, pool_bytes=64 * MiB) as c:
        cl = make_client(bb, c)
        # 3 MiB + 48 in 1 MiB-ish segments: the two shards split inside the second segment
        lens = [MiB + 16, MiB - 32, MiB + 64]
        src = Layout(lens, rng)
        cfg = cfg_for(bb, algo, replication_factor=2, max_workers_per_copy=2)
        assert cl.batch_put_device_gather(["st"], src.segs, [3], cfg, 0) == [bb.ErrorCode.OK]
        copies = cl.get_workers("st")
        assert len(copies) == 2 and all(len(cp.shards) == 2 for cp in copies)
        blob = np.frombuffer(src.concat(), dtype=np.uint8)
        off = 0
        for sh0, sh1 in zip(copies[0].shards, copies[1].shards):
            ref = blob[off:off + sh0.length]
            want = bb.bbh64_reference(ref) if algo == "BBH64" else bb.crc32c(ref)
            assert sh0.checksum == want == sh1.checksum
            off += sh0.length
        assert copies[0].shards[0].length not in (lens[0], lens[0] + lens[1])  # the boundary is inside a segment
        # corrupt one replica's first shard: the scattered get fails over to the other copy
        pools = {p.id: p for p in cl.keystone().get_memory_pools()}
        for cp in copies[:1]:
            sh = cp.shards[0]
            w = [w for w in c.workers if w.backend(sh.pool_id) is not None][0]
            o = sh.location["remote_addr"] - pools[sh.pool_id].ucx_remote_addr + 5
            w.backend(sh.pool_id).write(o, bytes([w.backend(sh.pool_id).read(o, 1)[0] ^ 0xFF]))
        for _ in range(2):  # whichever replica the client picks first
            dst = Layout(split(blob.size, rng, 256 * 1024), rng, fill_random=False)
            assert cl.batch_get_device_scatter(["st"], dst.segs, [len(dst.lens)], 0) == [bb.ErrorCode.OK]
            assert dst.concat() == blob.tobytes() and dst.guards_intact()


def test_host_tier_objects_take_the_staged_path_both_ways(bb, tmp_path):
    rng = np.random.default_rng(5)
    with LocalCluster(cluster_id="seg-stage", n_workers=1, pool_bytes=64 * MiB) as c:
        c.keystone.install_data_server_mover()
        c.add_worker("worker-disk", "node-9", [("disk-0", bb.StorageClass.NVME, 64 * MiB, str(tmp_path))])
        cl = make_client(bb, c, reach_disk=False)
        objs = [split(150_000, rng, 4096), [4096] * 7 + [5]]
        src = Layout([x for o in objs for x in o], rng)
        counts = [len(o) for o in objs]
        nv = cfg_for(bb, "CRC32C", preferred_classes=[bb.StorageClass.NVME])
        assert cl.batch_put_device_gather(["h/0", "h/1"], src.segs, counts, nv, 0) == [bb.ErrorCode.OK] * 2
        assert cl.get_workers("h/0")[0].shards[0].storage_class == bb.StorageClass.NVME
        ram = cfg_for(bb, "BBH64")
        assert cl.batch_put_device_gather(["h/2"], src.segs[:counts[0]], [counts[0]], ram, 0) == [bb.ErrorCode.OK]
        assert cl.migrate("h/2", bb.StorageClass.NVME) == bb.ErrorCode.OK  # demoted to a tier the transport cannot reach
        assert cl.get_workers("h/2")[0].shards[0].storage_class == bb.StorageClass.NVME
        keys = ["h/0", "h/1", "h/2"]
        totals = [sum(objs[0]), sum(objs[1]), sum(objs[0])]
        dobjs = [split(t, rng, 2048) for t in totals]
        dst = Layout([x for o in dobjs for x in o], rng, fill_random=False)
        assert cl.batch_get_device_scatter(keys, dst.segs, [len(o) for o in dobjs], 0) == [bb.ErrorCode.OK] * 3
        d = 0
        for i, want in enumerate([src.concat(0, counts[0]), src.concat(counts[0], counts[1]), src.concat(0, counts[0])]):
            assert dst.concat(d, len(dobjs[i])) == want
            d += len(dobjs[i])
        assert dst.guards_intact()
        m = cl.metrics_text()
        assert "device_put_host_staged_total" in m and "device_get_host_staged_total" in m


def test_chunked_mixed_batch_and_the_segment_bound_per_launch(bb):
    rng = np.random.default_rng(6)
    with LocalCluster(cluster_id="seg-chunk", n_workers=2, pool_bytes=128 * MiB) as c:
        cl = make_client(bb, c)
        cl.set_device_pipeline_chunks(3)
        # three objects of 400k 16-byte segments: 1.2 M segments, more than one launch may carry
        big = [[16] * 400_000 for _ in range(3)]
        small = [[4096, 4096, 9], split(100_000, rng)]
        objs = [big[0], small[0], big[1], small[1], big[2]]
        buf = np.frombuffer(os.urandom(sum(sum(o) for o in objs) + 4096), dtype=np.uint8).copy()
        base = buf.ctypes.data + (-buf.ctypes.data) % 16
        boff = base - buf.ctypes.data
        rows, pos = [], 0
        for o in objs:
            for n in o:
                rows.append((base + pos, n))
                buf[boff + pos + n:boff + pos + (n + 15) // 16 * 16] = 0  # padding: not part of any object
                pos += (n + 15) // 16 * 16
        segs = np.array(rows, dtype=np.uint64)
        counts = [len(o) for o in objs]
        keys = [f"ch/{i}" for i in range(len(objs))]
        assert cl.batch_put_device_gather(keys, segs, counts, cfg_for(bb, "XXH3"), 0) == [bb.ErrorCode.OK] * len(keys)
        out = np.zeros(pos + 64, dtype=np.uint8)
        obase = out.ctypes.data + (-out.ctypes.data) % 16
        osegs = segs.copy()
        osegs[:, 0] = osegs[:, 0] - np.uint64(base) + np.uint64(obase)
        assert cl.batch_get_device_scatter(keys, osegs, counts, 0) == [bb.ErrorCode.OK] * len(keys)
        ooff = obase - out.ctypes.data
        assert np.array_equal(out[ooff:ooff + pos], buf[boff:boff + pos])
        for k, o in zip(keys, objs):
            assert sum(sh.length for sh in cl.get_workers(k)[0].shards) == sum(o)


def test_invalid_objects_are_rejected_one_by_one(bb):
    rng = np.random.default_rng(7)
    with LocalCluster(cluster_id="seg-valid", n_workers=1, pool_bytes=64 * MiB) as c:
        cl = make_client(bb, c)
        cfg = cfg_for(bb, "BBH64")
        good = Layout([4096, 4096, 100], rng)
        bad = Layout([4096, 4096, 100], rng)
        segs = np.concatenate([good.segs, bad.segs])
        cases = {
            "misaligned": lambda s: s.__setitem__((3, 0), s[3, 0] + np.uint64(8)),
            "odd-middle": lambda s: s.__setitem__((3, 1), np.uint64(4008)),
            "zero-length": lambda s: s.__setitem__((4, 1), np.uint64(0)),
        }
        for name, spoil in cases.items():
            s = segs.copy()
            spoil(s)
            ecs = cl.batch_put_device_gather([f"ok/{name}", f"bad/{name}"], s, [3, 3], cfg, 0)
            assert ecs == [bb.ErrorCode.OK, bb.ErrorCode.INVALID_PARAMETERS], name
            assert cl.object_exists(f"ok/{name}") and not cl.object_exists(f"bad/{name}")
        # empty object
        assert cl.batch_put_device_gather(["e/0", "e/1"], good.segs, [0, 3], cfg, 0) == [bb.ErrorCode.INVALID_PARAMETERS, bb.ErrorCode.OK]
        # seg_counts that do not add up to the table: the whole batch
        assert cl.batch_put_device_gather(["w/0", "w/1"], segs, [3, 2], cfg, 0) == [bb.ErrorCode.INVALID_PARAMETERS] * 2
        assert not cl.object_exists("w/0")
        # get: a list that does not cover the stored size exactly writes nothing for that object
        dst = Layout([4096, 4096, 100], rng, fill_random=False)
        short = Layout([4096, 4096, 99], rng, fill_random=False)
        before = short.buf.copy()
        ecs = cl.batch_get_device_scatter(["ok/misaligned", "e/1"], np.concatenate([short.segs, dst.segs]), [3, 3], 0)
        assert ecs == [bb.ErrorCode.INVALID_PARAMETERS, bb.ErrorCode.OK]
        assert np.array_equal(short.buf, before) and dst.concat() == good.concat()
        # and the per-object rules on get
        s = np.concatenate([dst.segs, short.segs])
        s[1, 1] = np.uint64(4008)
        assert cl.batch_get_device_scatter(["e/1"], s[:3], [3], 0) == [bb.ErrorCode.INVALID_PARAMETERS]


def test_segment_tables_from_numpy_and_torch(bb):
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(8)
    with LocalCluster(cluster_id="seg-types", n_workers=1, pool_bytes=32 * MiB) as c:
        cl = make_client(bb, c)
        src = Layout([4096, 4096, 77], rng)
        cfg = cfg_for(bb, "XXH3")
        assert cl.batch_put_device_gather(["np"], src.segs, [3], cfg, 0) == [bb.ErrorCode.OK]
        assert cl.batch_put_device_gather(["np64"], src.segs.astype(np.int64), [3], cfg, 0) == [bb.ErrorCode.OK]
        assert cl.batch_put_device_gather(["pt"], torch.from_numpy(src.segs.astype(np.int64)), [3], cfg, 0) == [bb.ErrorCode.OK]
        dst = Layout([8192, 77], rng, fill_random=False)
        for k in ("np", "np64", "pt"):
            dst.buf[dst.mask] = 0
            assert cl.batch_get_device_scatter([k], torch.from_numpy(dst.segs.astype(np.int64)), [2], 0) == [bb.ErrorCode.OK]
            assert dst.concat() == src.concat()
        with pytest.raises((TypeError, ValueError)):
            cl.batch_put_device_gather(["x"], src.segs[:, :1].copy(), [3], cfg, 0)
        with pytest.raises((TypeError, ValueError)):
            cl.batch_put_device_gather(["x"], src.segs.astype(np.float64), [3], cfg, 0)
