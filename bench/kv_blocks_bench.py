#!/usr/bin/env python3
"""Paged-KV block offload on one GPU: four ways to store and load the same chunk of a paged KV cache.

Layout: 80 layers x (K, V) = 160 cache tensors [num_blocks, block_bytes] (bf16), 16 objects (sequence chunks) of 16
blocks per layer and kind, i.e. 2560 segments per object.  At 32 KiB blocks an object is 80 MiB and a batch 1.25 GiB
(larger than L2).  Repeated with 4 KiB and 16 KiB blocks.

  (a) blocks   TensorStore-style gather put / scatter get (batch_put_device_gather / batch_get_device_scatter)
  (b) staging  gather into a staging tensor + batch_put_device; batch_get_device + scatter out of it (public API today)
  (c) per-block one object per block through batch_put_device / batch_get_device
  (d) ceiling  contiguous put / get of an equally sized buffer

For every arm: wall time of whole calls (host clock around the call, ending in a device synchronise) and kernel time
(fabric.total_device_ms).  With --trace, per-tile pipeline timestamps of one (a) and one (d) put are summarised.
Writes <outdir>/kv_blocks.json with the card name and power limit.

    python bench/kv_blocks_bench.py OUTDIR [--iters 3] [--blocks-kib 4 16 32] [--trace]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from blackbird_b200 import _bb  # noqa: E402
from blackbird_b200.parallel import GpuRankCluster  # noqa: E402

LAYERS, KINDS, NOBJ, BLOCKS_PER = 80, 2, 16, 16


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    name, _, power = line.partition(",")
    return {"name": name.strip() or torch.cuda.get_device_name(0), "power_limit": power.strip() or "unknown"}


def timed(cl, fn):
    torch.cuda.synchronize()
    k0 = cl.fabric.total_device_ms
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3, cl.fabric.total_device_ms - k0


def trace_summary(tr):
    t = np.array(tr, dtype=np.int64).reshape(-1, 4)
    t = t[(t > 0).all(1)]
    if len(t) == 0:
        return None
    return {"tiles": int(len(t)), "span_us": float((t[:, 3].max() - t[:, 0].min()) / 1e3),
            "load_issue_to_landed_us_p50": float(np.median(t[:, 1] - t[:, 0]) / 1e3),
            "landed_to_store_issued_us_p50": float(np.median(t[:, 2] - t[:, 1]) / 1e3),
            "store_issued_to_released_us_p50": float(np.median(t[:, 3] - t[:, 2]) / 1e3)}


def run_config(cl, block_kib, iters, do_trace):
    dev = torch.device("cuda", cl.local_rank)
    s = torch.cuda.current_stream().cuda_stream
    block = block_kib * 1024
    nblocks = NOBJ * BLOCKS_PER + 8
    caches = [torch.randint(-1000, 1000, (nblocks, block // 2), dtype=torch.int16, device=dev).view(torch.bfloat16)
              for _ in range(LAYERS * KINDS)]
    ncache = len(caches)
    g = torch.Generator().manual_seed(block_kib)
    perm = torch.randperm(nblocks, generator=g)[:NOBJ * BLOCKS_PER]
    ids = perm.view(NOBJ, BLOCKS_PER)
    obj_bytes = ncache * BLOCKS_PER * block
    total = NOBJ * obj_bytes
    cfg = _bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1, ttl_ms=0, preferred_classes=[_bb.StorageClass.RAM_GPU],
                           checksum=_bb.ChecksumAlgo.XXH3)
    # segment table: object i = cache by cache, blocks ids[i]
    bases = torch.tensor([c.data_ptr() for c in caches], dtype=torch.int64)[:, None]
    rows = [torch.stack([(bases + ids[i][None, :] * block).reshape(-1), torch.full((ncache * BLOCKS_PER,), block, dtype=torch.int64)], 1)
            for i in range(NOBJ)]
    segs = torch.cat(rows).numpy()
    counts = [ncache * BLOCKS_PER] * NOBJ
    ids_dev = ids.to(dev)
    flat_ids = ids_dev.reshape(-1)
    results = {"block_kib": block_kib, "segments_per_object": counts[0], "object_mib": obj_bytes / 2**20, "batch_gib": total / 2**30}

    def arm(name, put, get, keys):
        put_w, put_k, get_w, get_k = [], [], [], []
        for it in range(iters + 1):  # the first pass warms up
            ecs, w, k = timed(cl, put)
            assert all(e == _bb.ErrorCode.OK for e in ecs), (name, ecs[:3])
            ecs, w2, k2 = timed(cl, get)
            assert all(e == _bb.ErrorCode.OK for e in ecs), (name, ecs[:3])
            cl.client.batch_remove(keys)
            if it:
                put_w.append(w), put_k.append(k), get_w.append(w2), get_k.append(k2)
        med = statistics.median
        results[name] = {"put_call_ms": med(put_w), "put_kernel_ms": med(put_k), "get_call_ms": med(get_w), "get_kernel_ms": med(get_k),
                         "put_call_GBps": total / med(put_w) / 1e6, "get_call_GBps": total / med(get_w) / 1e6,
                         "put_kernel_GBps": total / med(put_k) / 1e6 if med(put_k) else None,
                         "get_kernel_GBps": total / med(get_k) / 1e6 if med(get_k) else None}

    keys = [f"kvb/{block_kib}/{i}" for i in range(NOBJ)]
    ref = [c[ids_dev[3]].clone() for c in caches[:4]]
    arm("a_blocks", lambda: cl.client.batch_put_device_gather(keys, segs, counts, cfg, s),
        lambda: cl.client.batch_get_device_scatter(keys, segs, counts, s), keys)
    assert all(torch.equal(c[ids_dev[3]].view(torch.int16), r.view(torch.int16)) for c, r in zip(caches[:4], ref))

    staging = torch.empty((NOBJ, ncache, BLOCKS_PER, block // 2), dtype=torch.bfloat16, device=dev)

    def put_b():
        for ci, c in enumerate(caches):
            staging[:, ci] = c[ids_dev]
        return cl.client.batch_put_device(keys, [staging[i].data_ptr() for i in range(NOBJ)], [obj_bytes] * NOBJ, cfg, s)

    def get_b():
        ecs, _ = cl.client.batch_get_device(keys, [staging[i].data_ptr() for i in range(NOBJ)], [obj_bytes] * NOBJ, s)
        for ci, c in enumerate(caches):
            c.index_copy_(0, flat_ids, staging[:, ci].reshape(-1, block // 2))
        return ecs

    arm("b_staging", put_b, get_b, keys)
    del staging
    torch.cuda.empty_cache()

    bkeys = [f"kvb1/{block_kib}/{j}" for j in range(NOBJ * ncache * BLOCKS_PER)]
    bptr = segs[:, 0].tolist()
    arm("c_per_block", lambda: cl.client.batch_put_device(bkeys, bptr, [block] * len(bkeys), cfg, s),
        lambda: cl.client.batch_get_device(bkeys, bptr, [block] * len(bkeys), s)[0], bkeys)

    flat = torch.randint(0, 256, (total,), dtype=torch.uint8, device=dev)
    fptr = [flat.data_ptr() + i * obj_bytes for i in range(NOBJ)]
    arm("d_contiguous", lambda: cl.client.batch_put_device(keys, fptr, [obj_bytes] * NOBJ, cfg, s),
        lambda: cl.client.batch_get_device(keys, fptr, [obj_bytes] * NOBJ, s)[0], keys)

    if do_trace:
        tr = {}
        for name, put in (("a_blocks", lambda: cl.client.batch_put_device_gather(keys, segs, counts, cfg, s)),
                          ("d_contiguous", lambda: cl.client.batch_put_device(keys, fptr, [obj_bytes] * NOBJ, cfg, s))):
            cl.fabric.set_tile_trace(True)
            timed(cl, put)
            cl.fabric.set_tile_trace(False)
            tr[name] = trace_summary(cl.fabric.tile_trace())
            cl.client.batch_remove(keys)
        results["tile_trace_put"] = tr
    a, d = results["a_blocks"], results["d_contiguous"]
    results["a_over_d_kernel"] = {"put": d["put_kernel_ms"] / a["put_kernel_ms"], "get": d["get_kernel_ms"] / a["get_kernel_ms"]}
    del caches, flat
    torch.cuda.empty_cache()
    return results


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--blocks-kib", type=int, nargs="+", default=[4, 16, 32])
    ap.add_argument("--trace", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("kv_blocks_bench needs a GPU")
    os.makedirs(a.outdir, exist_ok=True)
    cl = GpuRankCluster(slab_bytes=3 << 30, cluster_id="kvbench")
    try:
        out = {"card": card(), "layers": LAYERS, "objects": NOBJ, "blocks_per_object_per_cache": BLOCKS_PER, "checksum": "XXH3",
               "configs": [run_config(cl, b, a.iters, a.trace) for b in a.blocks_kib]}
    finally:
        cl.stop()
    with open(os.path.join(a.outdir, "kv_blocks.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
