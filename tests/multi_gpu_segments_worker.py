"""Rank program of tests/test_gpu_segments.py::test_segments_across_gpus (torchrun, one rank per GPU).

Segmented objects on N >= 2 GPUs: blocks of this rank's paged-KV caches gathered into an object placed on the ring
neighbour's HBM (NVLink), scattered back into other blocks, and -- when an NVLS group exists -- gathered into symmetric
replicas (one multimem.st stream per object).  Prints one JSON line per rank; an assertion failure fails torchrun."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if os.environ.get("BB_PKG_ROOT"):
    sys.path.insert(0, os.path.abspath(os.environ["BB_PKG_ROOT"]))
from blackbird_b200 import _bb  # noqa: E402
from blackbird_b200.ops.tensor_store import TensorStore  # noqa: E402
from blackbird_b200.parallel import GpuRankCluster  # noqa: E402


def main():
    world_env = int(os.environ.get("WORLD_SIZE", "1"))
    cl = GpuRankCluster(slab_bytes=512 << 20, cluster_id="t-multi-seg", nvls_arena_bytes=128 << 20, nvls_group_size=min(3, world_env))
    rank, world = cl.rank, cl.world
    nxt = (rank + 1) % world
    dev = torch.device("cuda", cl.local_rank)
    torch.cuda.set_device(dev)
    res = {"rank": rank, "world": world}
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    caches = [torch.randn((32, 16, 8, 128), generator=g, device=dev).to(torch.bfloat16) for _ in range(8)]
    orig = [c.clone() for c in caches]
    keys = [f"mseg/{rank}/{i}" for i in range(4)]
    put_ids = [torch.arange(i * 6, i * 6 + 6) for i in range(4)]
    get_ids = [torch.arange(31 - i * 6, 25 - i * 6, -1) for i in range(4)]

    for algo in (_bb.ChecksumAlgo.BBH64, _bb.ChecksumAlgo.CRC32C):
        cfg = _bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1, preferred_node=f"gpu{nxt}", ttl_ms=0, checksum=algo,
                               preferred_classes=[_bb.StorageClass.RAM_GPU])
        store = TensorStore(cl.client, cfg)
        store.batch_put_blocks(keys, caches, put_ids)
        sh = cl.client.get_workers(keys[1])[0].shards[0]
        assert sh.worker_id == f"worker-gpu{nxt}", sh.worker_id
        want = torch.cat([o[put_ids[1]].reshape(-1).view(torch.uint8) for o in orig])
        ref = want.cpu().numpy()
        assert sh.checksum == (_bb.bbh64(ref) if algo == _bb.ChecksumAlgo.BBH64 else _bb.crc32c(ref))
        for c in caches:
            c.zero_()
        store.batch_get_blocks(keys, caches, get_ids)
        torch.cuda.synchronize()
        for i in range(4):
            assert all(torch.equal(c[get_ids[i]].view(torch.int16), o[put_ids[i]].view(torch.int16)) for c, o in zip(caches, orig))
        store.remove(keys)
        for c, o in zip(caches, orig):
            c.copy_(o)
    res["ring"] = "ok"
    assert cl.fabric.path_bytes(True, 1) > 0 and cl.fabric.path_bytes(False, 1) > 0
    cl.barrier()

    if cl.arena is not None:
        R = min(3, world)
        before = cl.fabric.multicast_puts
        cfg = _bb.WorkerConfig(replication_factor=R, max_workers_per_copy=1, ttl_ms=0, symmetric_replicas=True,
                               preferred_classes=[_bb.StorageClass.RAM_GPU])
        store = TensorStore(cl.client, cfg)
        store.batch_put_blocks(keys, caches, put_ids)
        res["nvls_multicast"] = cl.fabric.multicast_puts > before
        for c in caches:
            c.zero_()
        store.batch_get_blocks(keys, caches, get_ids)
        torch.cuda.synchronize()
        for i in range(4):
            assert all(torch.equal(c[get_ids[i]].view(torch.int16), o[put_ids[i]].view(torch.int16)) for c, o in zip(caches, orig))
        store.remove(keys)
    cl.barrier()
    cl.stop()
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
