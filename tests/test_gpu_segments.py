"""GPU tests of segmented objects: the gather / scatter variant of the fused kernel against contiguous transfers of the
same bytes (engine level), the paged-KV block API of TensorStore on the full stack, and the multi-GPU data plane
(tests/multi_gpu_segments_worker.py under torchrun, skipped on one GPU)."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GUARD = 0xAB
KiB = 1024


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.fail("GPU tests need CUDA (marked gpu)")
    return torch


def _stream(torch):
    return torch.cuda.current_stream().cuda_stream


class DevLayout:
    """Segments of the given lengths at shuffled 16-byte aligned places of one device buffer, separated by guard
    bytes.  tables[i] = (S_i, 2) int64 table of object i."""

    def __init__(self, torch, objs, rng, fill_random):
        lens = [n for o in objs for n in o]
        slot = [(n + 15) // 16 * 16 + 32 for n in lens]
        total = sum(slot) + 64
        self.buf = torch.full((total,), GUARD, dtype=torch.uint8, device="cuda")
        order = rng.permutation(len(lens))
        starts, pos = [0] * len(lens), 32
        for k in order:
            starts[k] = pos
            pos += slot[k]
        mask = np.zeros(total, dtype=bool)
        for s, n in zip(starts, lens):
            mask[s:s + n] = True
        self.mask = torch.from_numpy(mask).cuda()
        if fill_random:
            rnd = torch.randint(0, 256, (total,), dtype=torch.uint8, device="cuda")
            self.buf[self.mask] = rnd[self.mask]
        base = self.buf.data_ptr()
        self.tables, self.pieces, k = [], [], 0
        for o in objs:
            idx = range(k, k + len(o))
            self.tables.append(np.array([[base + starts[j], lens[j]] for j in idx], dtype=np.int64).reshape(-1, 2))
            self.pieces.append([(starts[j], lens[j]) for j in idx])
            k += len(o)

    def concat(self, torch, i):
        return torch.cat([self.buf[s:s + n] for s, n in self.pieces[i]])

    def guards_intact(self):
        return bool((self.buf[~self.mask] == GUARD).all())


def mix(name, rng, nobj):
    """Segment lengths per object for one segment-size mix."""
    small = nobj > 8
    if name == "16B":
        return [[16] * (64 if small else 1024) for _ in range(nobj)]
    if name == "4K":
        return [[4 * KiB] * (5 if small else 40) for _ in range(nobj)]
    if name == "32K":
        return [[32 * KiB] * (2 if small else 12) for _ in range(nobj)]
    if name == "random":
        return [[int(x) * 16 for x in rng.integers(1, 200 * KiB // 16 + 1, 2 if small else 8)] for _ in range(nobj)]
    if name == "span":  # one segment spanning many tiles between small ones
        return [[48, (9 * 16 * KiB if small else 40 * 16 * KiB) + 32, 16] for _ in range(nobj)]
    if name == "tail":  # last segment with a 1-15 byte tail
        return [[4 * KiB, 16 * KiB + 48, int(rng.integers(0, 64)) * 16 + 1 + i % 15] for i in range(nobj)]
    raise ValueError(name)


MIXES = ["16B", "4K", "32K", "random", "span", "tail"]


@pytest.mark.parametrize("ctas", [1, 2, 5, 0])
@pytest.mark.parametrize("algo_name", ["XXH3", "CRC32C", "BBH64", "NONE"])
def test_segmented_items_match_contiguous_items(bb, torch_cuda, algo_name, ctas):
    torch = torch_cuda
    algo = getattr(bb.ChecksumAlgo, algo_name)
    rng = np.random.default_rng(1000 + ctas)
    eng = bb.XferEngine(0, 1024, 2)
    eng.set_max_ctas(ctas)
    s = _stream(torch)
    for nobj in (1, 8, 300):
        for name in MIXES:
            objs = mix(name, rng, nobj)
            sizes = [sum(o) for o in objs]
            offs = np.cumsum([0] + [(n + 255) // 256 * 256 for n in sizes]).tolist()
            src = DevLayout(torch, objs, rng, True)
            concat = [src.concat(torch, i) for i in range(nobj)]
            slab_g = torch.zeros(offs[-1], dtype=torch.uint8, device="cuda")
            slab_c = torch.zeros(offs[-1], dtype=torch.uint8, device="cuda")
            dg_g, _, _ = eng.run([(src.tables[i], slab_g.data_ptr() + offs[i], sizes[i]) for i in range(nobj)], algo, s)
            dg_c, _, _ = eng.run([(concat[i].data_ptr(), slab_c.data_ptr() + offs[i], sizes[i]) for i in range(nobj)], algo, s)
            torch.cuda.synchronize()
            assert dg_g == dg_c, (name, nobj)
            assert torch.equal(slab_g, slab_c), (name, nobj)
            # scatter back into a different split of the same sizes
            dobjs = [[16 * KiB] * (n // (16 * KiB)) + ([n % (16 * KiB)] if n % (16 * KiB) else []) if i % 2 else o
                     for i, (o, n) in enumerate(zip(objs, sizes))]
            dst = DevLayout(torch, dobjs, rng, False)
            flags = bb.XFER_VERIFY if algo_name != "NONE" else 0
            _, st, _ = eng.run([(slab_g.data_ptr() + offs[i], dst.tables[i], sizes[i], dg_g[i], flags) for i in range(nobj)], algo, s)
            torch.cuda.synchronize()
            assert st == [0] * nobj, (name, nobj)
            for i in range(nobj):
                assert torch.equal(dst.concat(torch, i), concat[i]), (name, nobj, i)
            assert dst.guards_intact() and src.guards_intact(), (name, nobj)
            if algo_name != "NONE":  # a flipped stored byte flags exactly its object
                bad = nobj // 2
                slab_g[offs[bad] + sizes[bad] // 2] ^= 0x40
                _, st, _ = eng.run([(slab_g.data_ptr() + offs[i], dst.tables[i], sizes[i], dg_g[i], flags) for i in range(nobj)], algo, s)
                torch.cuda.synchronize()
                assert st == [1 if i == bad else 0 for i in range(nobj)], (name, nobj)


@pytest.mark.parametrize("nrep", [1, 2, 3])
def test_gather_fans_out_to_replicas(bb, torch_cuda, nrep):
    torch = torch_cuda
    rng = np.random.default_rng(7 + nrep)
    eng = bb.XferEngine(0, 1024, 2)
    objs = mix("random", rng, 8) + mix("tail", rng, 4)
    sizes = [sum(o) for o in objs]
    offs = np.cumsum([0] + [(n + 255) // 256 * 256 for n in sizes]).tolist()
    src = DevLayout(torch, objs, rng, True)
    reps = [torch.zeros(offs[-1], dtype=torch.uint8, device="cuda") for _ in range(nrep)]
    dg, _, _ = eng.run([(src.tables[i], [r.data_ptr() + offs[i] for r in reps], sizes[i]) for i in range(len(objs))],
                       bb.ChecksumAlgo.BBH64, _stream(torch))
    torch.cuda.synchronize()
    for i in range(len(objs)):
        want = src.concat(torch, i)
        assert dg[i] == bb.bbh64(want.cpu().numpy())
        assert all(torch.equal(r[offs[i]:offs[i] + sizes[i]], want) for r in reps)


def _paged_kv(torch, layers=8, blocks=64):
    g = torch.Generator(device="cuda").manual_seed(5)
    return [torch.randn((blocks, 16, 8, 128), generator=g, device="cuda").to(torch.bfloat16) for _ in range(2 * layers)]


def test_paged_kv_blocks_full_stack(bb, torch_cuda):
    torch = torch_cuda
    from blackbird_b200.ops.tensor_store import TensorStore
    from blackbird_b200.parallel import GpuRankCluster

    cl = GpuRankCluster(slab_bytes=512 << 20, cluster_id="t-kvblocks", dram_bytes=128 << 20)
    try:
        store = TensorStore(cl.client)
        caches = _paged_kv(torch)
        orig = [c.clone() for c in caches]
        perm = torch.randperm(64)
        keys = [f"kv/{i}" for i in range(6)]
        put_ids = [perm[i * 8:(i + 1) * 8] for i in range(6)]
        store.batch_put_blocks(keys, caches, put_ids)
        torch.cuda.synchronize()
        # store.get sees the concatenation of the blocks (cache by cache)
        flat = store.get(keys[2])
        want = torch.cat([c[put_ids[2]].reshape(-1).view(torch.uint8) for c in orig])
        assert flat.dtype == torch.uint8 and torch.equal(flat, want)
        for c in caches:
            c.zero_()
        perm2 = torch.randperm(64)
        get_ids = [perm2[i * 8:(i + 1) * 8] for i in range(6)]
        store.batch_get_blocks(keys, caches, get_ids)
        torch.cuda.synchronize()
        for i in range(6):
            for c, o in zip(caches, orig):
                assert torch.equal(c[get_ids[i]].view(torch.int16), o[put_ids[i]].view(torch.int16))
        untouched = torch.ones(64, dtype=torch.bool)
        untouched[torch.cat(get_ids)] = False
        assert all(bool((c[untouched].view(torch.int16) == 0).all()) for c in caches)
        # a key demoted to the DRAM tier still scatters back
        assert cl.client.migrate(keys[4], bb.StorageClass.RAM_CPU) == bb.ErrorCode.OK
        assert cl.client.get_workers(keys[4])[0].shards[0].storage_class == bb.StorageClass.RAM_CPU
        for c in caches:
            c[get_ids[4]] = 0
        store.batch_get_blocks([keys[4]], caches, [get_ids[4]])
        torch.cuda.synchronize()
        assert all(torch.equal(c[get_ids[4]].view(torch.int16), o[put_ids[4]].view(torch.int16)) for c, o in zip(caches, orig))
        store.remove(keys)
        assert not any(cl.client.object_exists(k) for k in keys)
    finally:
        cl.stop()


def test_small_segmented_objects_take_the_big_kernel(bb, torch_cuda):
    torch = torch_cuda
    from blackbird_b200.parallel import GpuRankCluster

    cl = GpuRankCluster(slab_bytes=64 << 20, cluster_id="t-segsmall")
    try:
        rng = np.random.default_rng(11)
        objs = [[16 * (1 + i), 256, 48 + i] for i in range(8)]  # each well under 4 KiB
        src = DevLayout(torch, objs, rng, True)
        segs = np.concatenate(src.tables)
        counts = [len(o) for o in objs]
        keys = [f"ss/{i}" for i in range(8)]
        s = _stream(torch)
        cfg = bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1, preferred_classes=[bb.StorageClass.RAM_GPU],
                              checksum=bb.ChecksumAlgo.CRC32C)
        small0, l0 = cl.fabric.small_launches, cl.fabric.launches
        assert cl.client.batch_put_device_gather(keys, segs, counts, cfg, s) == [bb.ErrorCode.OK] * 8
        dst = DevLayout(torch, [[sum(o)] for o in objs], rng, False)  # one (unaligned-length) segment per object
        assert cl.client.batch_get_device_scatter(keys, np.concatenate(dst.tables), [len(t) for t in dst.tables], s) == [bb.ErrorCode.OK] * 8
        torch.cuda.synchronize()
        assert cl.fabric.small_launches == small0 and cl.fabric.launches >= l0 + 2
        for i in range(8):
            want = src.concat(torch, i)
            assert torch.equal(dst.concat(torch, i), want)
            assert cl.client.get_workers(keys[i])[0].shards[0].checksum == bb.crc32c(want.cpu().numpy())
        assert dst.guards_intact()
    finally:
        cl.stop()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_segments_across_gpus(torch_cuda):
    n = torch_cuda.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    world = min(n, 4)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "multi_gpu_segments_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    lines = [json.loads(x) for x in r.stdout.splitlines() if x.startswith("{")]
    assert len(lines) == world and all(x["ring"] == "ok" for x in lines), lines
