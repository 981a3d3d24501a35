#!/usr/bin/env python3
"""Headline benchmark: batched put + get throughput of the object store on N B200 workers.

Metric (BASELINE.json): batched put/get GB/s (and p50 / p99 us) at 1/2/4/8 GPU-tier workers, synthetic random-byte
objects, device-timed, max over ranks.  One *step* = one `batch_put_device` of B objects of S bytes (fused kernel:
transfer + XXH3 digest, placements from the Keystone) followed by one `batch_get_device` of the same objects (fused
kernel: transfer + digest verify), then a `batch_remove` so that the slab is recycled.  `value` = payload bytes moved
per second by the whole job (put bytes + get bytes, all ranks).

Topology: one process per GPU (torchrun); rank 0 hosts the Keystone (RPC over loopback for the other ranks); every rank
runs a GPU-tier worker whose HBM slab is exported to all peers (CUDA IPC).  With N >= 2 every object is placed on the
writer's ring neighbour, so every payload byte crosses NVLink once per put and once per get; with N = 1 the slab is local
(HBM-bound).  Ranks meet through a shared-memory rendezvous (no NCCL on the product's path; NCCL is initialised after
the timed regions, for the comparators only).

  python bench.py --gpus 1 --steps 20 --warmup 3
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29511 \\
      bench.py --gpus 8 --steps 20 --warmup 3
  python bench.py --config sweep|spill          (N = 1)      torchrun ... bench.py --gpus 8 --config repl3|fanout|sweep

`--config` selects the BASELINE.json workload: headline (config #2 at one object size, the default), sweep (config #2:
GB/s and p50/p99 per size), repl3 (config #3), spill (config #4), fanout (config #5).
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BASELINE_GBPS = 0.233  # the only throughput figure in the reference tree (configs/worker.yaml:19, unsourced)
NVLINK_NOMINAL_GBPS = 900.0  # BASELINE.json: per direction per GPU
DUMP_SAMPLE_BYTES = 8 << 20  # --dump-outputs: payload bytes sampled over all ranks, 32 MB as float32
DUMP_SEED = 0xB200


def reference_arm() -> int:
    """The reference cannot be installed or built offline (DESIGN.md section 3 records the attempts)."""
    why = ("blackbird-io/blackbird is a CMake C++ project with no Python package: `pip install --no-index --no-build-isolation "
           "--find-links /opt/wheelhouse --target baseline/_ref /root/reference` fails (neither setup.py nor pyproject.toml); cmake "
           "configure needs the network (yalantinglibs / GoogleTest FetchContent) and UCX, etcd-cpp-apiv3, glog, yaml-cpp, liburing "
           "which are absent here and on the GPU box (profiles/r2_nvlink/ucx_probe.txt: no ucx_info, no /opt/hpcx, no libucp); "
           "src/worker/storage/cxl_memory_backend.cpp does not compile at this commit; its GPU pools are std::malloc")
    if int(os.environ.get("RANK", "0")) == 0:  # one line for the job, also when launched under torchrun
        print(json.dumps({"impl": "reference", "unavailable": why}))
    return 0


def pct(v, q):
    v = sorted(v)
    return v[min(len(v) - 1, int(q * len(v)))]


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--ctas", type=int, default=0, help="persistent CTAs of the fused kernel (0 = default)")
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--config", default="headline", choices=["headline", "sweep", "repl3", "spill", "fanout"])
    ap.add_argument("--objects", type=int, default=64, help="objects per batch per rank")
    ap.add_argument("--object-mib", type=float, default=64.0)
    ap.add_argument("--algo", default="xxh3", choices=["xxh3", "crc32c", "bbh64", "none"],
                    help="digest fused into the transfer: xxh3 (default) = the standard XXH3-64 of every 16 KiB tile, combined order-independently; "
                         "crc32c = standard Castagnoli CRC of the object; bbh64 = the tensor-core hash")
    ap.add_argument("--e2e-steps", type=int, default=16,
                    help="steps of each end-to-end mode (8.6 GB over PCIe per step per rank); the pipelined mode pays one un-overlapped H2D at the start and one D2H at the end")
    ap.add_argument("--no-comparators", action="store_true")
    ap.add_argument("--sync", choices=["none", "step", "phase"], default="phase",
                    help="N>1: ranks rendezvous per step / per put-get phase (inside the timed region)")
    ap.add_argument("--idle-odd", action="store_true", help="diagnostic: odd ranks idle (unidirectional NVLink traffic)")
    ap.add_argument("--quick", action="store_true", help="sweep config: fewer sizes")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="headline config: after the timed steps, write what the last timed step handed back to its caller as DIR/<name>.npy "
                         "(a fixed sample of the bytes the get delivered, the get sizes, the put / get status codes)")
    args = ap.parse_args()
    if args.dump_outputs and args.config != "headline":
        ap.error("--dump-outputs applies to the headline config")
    if args.impl == "reference":
        return reference_arm()

    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and args.gpus > 1:
        print(f"bench.py: --gpus {args.gpus} needs torchrun with {args.gpus} ranks (WORLD_SIZE={world})", file=sys.stderr)
        return 2
    if args.config != "headline":
        return run_config(args, world)
    return run_headline(args, world)


# ====================================================================================================== headline
def run_headline(args, world: int) -> int:
    import numpy as np
    import torch

    from blackbird_b200 import _bb
    from blackbird_b200.models import latency_sweep
    from blackbird_b200.parallel import GpuRankCluster
    from blackbird_b200.utils import ClockSampler

    nobj = args.objects
    osz = int(args.object_mib * (1 << 20))
    step_bytes = nobj * osz
    ALGOS = {"xxh3": _bb.ChecksumAlgo.XXH3, "bbh64": _bb.ChecksumAlgo.BBH64, "crc32c": _bb.ChecksumAlgo.CRC32C, "none": _bb.ChecksumAlgo.NONE}
    algo = ALGOS[args.algo]

    cl = GpuRankCluster(slab_bytes=3 * step_bytes + (64 << 20))
    rank, dev = cl.rank, torch.device("cuda", cl.local_rank)
    stream = torch.cuda.current_stream().cuda_stream
    target_node = f"gpu{(rank + 1) % world}"  # ring neighbour (== self when N = 1)

    def cfg_for(a):
        return _bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1, preferred_node=target_node, ttl_ms=0, checksum=a,
                                preferred_classes=[_bb.StorageClass.RAM_GPU])

    cfg = cfg_for(algo)
    # synthetic random-byte objects: payload (1 GiB by default) is larger than L2 (126 MB)
    src = torch.empty(step_bytes, dtype=torch.uint8, device=dev)
    _bb.random_fill(src.data_ptr(), step_bytes, 0xB200 + rank, stream)
    out = torch.empty(step_bytes, dtype=torch.uint8, device=dev)
    src_ptrs = [src.data_ptr() + i * osz for i in range(nobj)]
    out_ptrs = [out.data_ptr() + i * osz for i in range(nobj)]
    sizes = [osz] * nobj
    OK = _bb.ErrorCode.OK
    idle = args.idle_odd and rank % 2 == 1

    def rendezvous():
        # inside the timed region: its cost is part of the reported number.  Host-side (shared memory): the client calls
        # are synchronous, so "every rank returned from its batch_put_device" is all a phase boundary has to establish.
        if world > 1:
            cl.host_barrier()

    def step(tag: str, i: int, keys=None, put_ptrs=None, get_ptrs=None, c=None):
        keys = keys or [f"r{rank}/{tag}{i}/o{j}" for j in range(nobj)]
        if args.sync != "none":
            rendezvous()  # bulk-synchronous step (checkpoint / KV hand-off pattern): all ranks put, then all ranks get
        if not idle:
            put_ecs = cl.client.batch_put_device(keys, put_ptrs or src_ptrs, sizes, c or cfg, stream)
            assert all(e == OK for e in put_ecs), f"put failed: {[str(e) for e in put_ecs if e != OK][:3]}"
        if args.sync == "phase":
            rendezvous()
        if not idle:
            get_ecs, got = cl.client.batch_get_device(keys, get_ptrs or out_ptrs, sizes, stream)
            assert all(e == OK for e in get_ecs), f"get failed: {[str(e) for e in get_ecs if e != OK][:3]}"
            ecs = cl.client.batch_remove(keys)
            assert all(e == OK for e in ecs)
            return put_ecs, get_ecs, got
        return None

    if args.ctas:
        cl.fabric.set_max_ctas(args.ctas)
    # ---------------------------------------------------------------- warm-up + correctness
    sampler = ClockSampler(cl.local_rank, 100).start() if rank == 0 else None
    warm = max(3, args.warmup)
    for i in range(warm):
        step("w", i)
    torch.cuda.synchronize()
    if not idle:
        assert torch.equal(src, out), "payload mismatch after put+get"

    # ---------------------------------------------------------------- device-resident timed region
    launches0 = cl.fabric.launches
    all_keys = [[f"r{rank}/t{i}/o{j}" for j in range(nobj)] for i in range(args.steps)]  # fresh keys every step
    cl.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        last = step("t", i, all_keys[i])
    e1.record()
    torch.cuda.synchronize()
    cl.barrier()
    ms = cl.max_over_ranks(e0.elapsed_time(e1))
    launches = int(cl.sum_over_ranks(cl.fabric.launches - launches0))
    dump = {}
    if args.dump_outputs and not idle:
        # Taken now because the phases below reuse `out`; written at the end.  The sample positions depend only on the
        # batch size, and the sources are seeded, so two builds run with the same arguments dump comparable arrays.
        put_ecs, get_ecs, got = last
        n_sample = min(step_bytes, DUMP_SAMPLE_BYTES // world)
        pick = np.sort(np.random.default_rng(DUMP_SEED).integers(0, step_bytes, n_sample)) if n_sample < step_bytes else np.arange(step_bytes)
        dump = {"get_bytes_sample": out[torch.from_numpy(pick).to(dev)].float(),
                "get_sizes": torch.tensor(got, dtype=torch.float64),
                "put_status": torch.tensor([int(e) for e in put_ecs], dtype=torch.float64),
                "get_status": torch.tensor([int(e) for e in get_ecs], dtype=torch.float64)}
    if ms < 1500:  # give nvidia-smi time to take samples under the same load (same count on every rank: steps rendezvous)
        for i in range(int(1200.0 / max(ms / args.steps, 0.05)) + 1):
            step("c", i)
    clocks = sampler.stop() if sampler else None
    phases = {k: round(v[1] / max(v[0], 1), 1) for k, v in cl.client.phase_summary().items() if k.startswith("phase_")}
    phases_max = {k: round(cl.max_over_ranks(phases.get(k, 0.0)), 1) for k in sorted(phases)} if world > 1 else phases
    total_bytes = 2.0 * step_bytes * args.steps * world
    value = total_bytes / (ms * 1e-3) / 1e9

    # kernel-only view of one put and one get per digest (explains the headline; the standard digest is the headline)
    variants = {}
    for name in ("xxh3", "crc32c", "bbh64", "none"):
        keys = [f"r{rank}/k-{name}/o{j}" for j in range(nobj)]
        if args.sync != "none":
            rendezvous()
        m0 = cl.fabric.total_device_ms
        assert all(e == OK for e in cl.client.batch_put_device(keys, src_ptrs, sizes, cfg_for(ALGOS[name]), stream))
        m1 = cl.fabric.total_device_ms
        if args.sync != "none":
            rendezvous()
        ecs, _ = cl.client.batch_get_device(keys, out_ptrs, sizes, stream)
        m2 = cl.fabric.total_device_ms
        cl.client.batch_remove(keys)
        pm, gm = cl.max_over_ranks(m1 - m0), cl.max_over_ranks(m2 - m1)  # sums of the (pipelined) chunk kernels
        variants[name] = {"put_ms": round(pm, 4), "get_ms": round(gm, 4), "put_GBps_per_gpu": round(step_bytes / pm / 1e6, 1),
                          "get_GBps_per_gpu": round(step_bytes / gm / 1e6, 1)}
    kernel_only = variants[args.algo]

    # ---------------------------------------------------------------- single-object latency (p50 / p99, whole client call)
    lat_rows = latency_sweep(cl, [256, 4096, 65536, 1 << 20], target_node, iters=200, algo=algo)
    latency = {}
    for r in lat_rows:
        latency[str(r["size"])] = {k: round(cl.max_over_ranks(r[k]), 1) for k in ("put_p50_us", "put_p99_us", "get_p50_us", "get_p99_us")}
    cl.barrier()

    # ---------------------------------------------------------------- end-to-end (pinned host -> store -> pinned host)
    # Every step: this step's inputs come from pinned host memory, and the WHOLE result of the get is back in pinned host
    # memory (and the digests / status words with it) before the step counts as done.
    h_src = torch.empty(step_bytes, dtype=torch.uint8).pin_memory()
    h_src.copy_(src.cpu())
    h_out = torch.zeros(step_bytes, dtype=torch.uint8).pin_memory()
    h_src_ptrs = [h_src.data_ptr() + i * osz for i in range(nobj)]
    h_out_ptrs = [h_out.data_ptr() + i * osz for i in range(nobj)]

    def e2e_step(i: int, zero_copy: bool):
        if zero_copy:
            # the fused kernels touch host memory themselves: the put pulls the pinned source over PCIe (the H2D copy IS
            # the put), the get stores straight into the pinned destination (the D2H copy IS the get)
            step("z", i, put_ptrs=h_src_ptrs, get_ptrs=h_out_ptrs)
        else:
            src.copy_(h_src, non_blocking=True)      # H2D of this step's inputs from pinned memory (copy engine)
            step("e", i)                               # public API: batch_put_device / batch_get_device
            h_out.copy_(out, non_blocking=True)      # D2H of the whole result
        torch.cuda.synchronize()

    def e2e_run(zero_copy: bool):
        h_out.zero_()
        out.zero_()
        e2e_step(-1, zero_copy)
        cl.barrier()
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e2.record()
        for i in range(args.e2e_steps):
            e2e_step(i, zero_copy)
        e3.record()
        torch.cuda.synchronize()
        cl.barrier()
        if not idle:
            assert torch.equal(h_out, h_src), "end-to-end payload mismatch (host copy of the get result != host source)"
        return cl.max_over_ranks(e2.elapsed_time(e3))

    def e2e_pipelined() -> float:
        """Same per-step contract (inputs H2D from pinned memory, whole result D2H into pinned memory), software-pipelined
        across steps with double buffers: while step i's put / get run on the main stream, step i+1's inputs are already
        coming in on a copy stream and step i-1's result is going out on another (PCIe is full duplex)."""
        srcs = [src, torch.empty_like(src)]
        outs = [out, torch.empty_like(out)]
        h_outs = [h_out, torch.zeros(step_bytes, dtype=torch.uint8).pin_memory()]
        s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
        main = torch.cuda.current_stream()
        ptrs = lambda t: [t.data_ptr() + i * osz for i in range(nobj)]

        def run(nsteps: int) -> None:
            ev_in = [None, None]
            with torch.cuda.stream(s_in):
                srcs[0].copy_(h_src, non_blocking=True)
                ev_in[0] = s_in.record_event()
            for i in range(nsteps):
                b = i % 2
                if i + 1 < nsteps:
                    with torch.cuda.stream(s_in):  # inputs of the NEXT step (its buffer was last read by the put of step i-1: done)
                        srcs[1 - b].copy_(h_src, non_blocking=True)
                        ev_in[1 - b] = s_in.record_event()
                main.wait_event(ev_in[b])
                s_out.synchronize() if i >= 2 else None  # outs[b] / h_outs[b] of step i-2 have left the device
                step("p", i, put_ptrs=ptrs(srcs[b]), get_ptrs=ptrs(outs[b]))  # synchronous: the result is in outs[b]
                with torch.cuda.stream(s_out):  # result of THIS step goes out while the next step runs
                    h_outs[b].copy_(outs[b], non_blocking=True)
            s_out.synchronize()

        for h in h_outs:
            h.zero_()
        run(2)
        torch.cuda.synchronize()
        cl.barrier()
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e2.record()
        run(args.e2e_steps)
        e3.record()
        torch.cuda.synchronize()
        cl.barrier()
        if not idle:
            assert all(torch.equal(h, h_src) for h in h_outs), "pipelined end-to-end payload mismatch"
        return cl.max_over_ranks(e2.elapsed_time(e3))

    e2e_staged_ms = e2e_run(False)
    e2e_zc_ms = e2e_run(True)
    e2e_pipe_ms = e2e_pipelined()
    e2e_mode, e2e_ms = min((("staged", e2e_staged_ms), ("zero_copy", e2e_zc_ms), ("pipelined", e2e_pipe_ms)), key=lambda t: t[1])
    e2e_value = 2.0 * step_bytes * args.e2e_steps * world / (e2e_ms * 1e-3) / 1e9
    tab = nobj * 64 + (nobj + 1) * 4
    h2d = step_bytes + 2 * tab          # payload + put / get descriptor tables
    d2h = step_bytes + 2 * nobj * 12    # whole get result + digests / status of put and get

    # ---------------------------------------------------------------- comparators (same buffers, outside the timed regions)
    comparators = {}
    if not args.no_comparators:
        def timed(fn, iters=5):
            fn()
            torch.cuda.synchronize()
            cl.barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(iters):
                fn()
            b.record()
            torch.cuda.synchronize()
            return cl.max_over_ranks(a.elapsed_time(b)) / iters

        scratch = torch.empty(step_bytes // 512 + 2, dtype=torch.int32, device=dev)
        crc = torch.zeros(1, dtype=torch.int32, device=dev)
        if world == 1:
            t = timed(lambda: [out[i * osz:(i + 1) * osz].copy_(src[i * osz:(i + 1) * osz]) for i in range(nobj)])
            comparators["per_object_cudaMemcpyAsync_GBps"] = round(step_bytes / t / 1e6, 1)

            def unfused():
                _bb.copy_simt(out.data_ptr(), src.data_ptr(), step_bytes, stream)
                _bb.crc32c_device(out.data_ptr(), step_bytes, crc.data_ptr(), scratch.data_ptr(), stream)

            t = timed(unfused, 2)
            comparators["unfused_copy_kernel_plus_crc32c_kernel_GBps"] = round(step_bytes / t / 1e6, 1)
        else:
            nxt_dev = (cl.local_rank + 1) % world  # single node: the ring neighbour's device ordinal
            peer = torch.empty(step_bytes, dtype=torch.uint8, device=torch.device("cuda", nxt_dev))  # this process's buffer ON the neighbour GPU
            torch.cuda.set_device(cl.local_rank)
            _bb.enable_peer_access(cl.local_rank, nxt_dev)
            cl.barrier()

            def memcpy_peer_objects():
                for i in range(nobj):
                    _bb.memcpy_peer_async(peer.data_ptr() + i * osz, nxt_dev, src_ptrs[i], cl.local_rank, osz, stream)

            def memcpy_peer_single():
                _bb.memcpy_peer_async(peer.data_ptr(), nxt_dev, src.data_ptr(), cl.local_rank, step_bytes, stream)

            def memcpy_peer_plus_crc():
                memcpy_peer_objects()
                _bb.crc32c_device(src.data_ptr(), step_bytes, crc.data_ptr(), scratch.data_ptr(), stream)

            t = timed(memcpy_peer_single)
            comparators["cudaMemcpyPeerAsync_single_copy_GBps_per_rank"] = round(step_bytes / t / 1e6, 1)  # measured P2P peak (copy engines, all ranks at once)
            t = timed(memcpy_peer_objects)
            comparators["per_object_cudaMemcpyPeerAsync_GBps_per_rank"] = round(step_bytes / t / 1e6, 1)
            t = timed(memcpy_peer_plus_crc, 3)
            comparators["unfused_memcpyPeer_plus_crc32c_kernel_GBps_per_rank"] = round(step_bytes / t / 1e6, 1)
            del peer
            # NCCL, only now.  It announces its version on fd 1 when the first communicator comes up: keep stdout for the
            # one JSON line (the announcement goes to stderr instead).
            sys.stdout.flush()
            saved_fd = os.dup(1)
            os.dup2(2, 1)
            dist = cl.ensure_dist()
            nxt, prv = (rank + 1) % world, (rank - 1) % world

            def nccl_objects():
                ops = []
                for i in range(nobj):
                    ops.append(dist.P2POp(dist.isend, src[i * osz:(i + 1) * osz], nxt))
                    ops.append(dist.P2POp(dist.irecv, out[i * osz:(i + 1) * osz], prv))
                for r in dist.batch_isend_irecv(ops):
                    r.wait()

            def nccl_single():
                for r in dist.batch_isend_irecv([dist.P2POp(dist.isend, src, nxt), dist.P2POp(dist.irecv, out, prv)]):
                    r.wait()

            t = timed(nccl_single, 3)
            comparators["nccl_send_recv_one_message_GBps_per_rank"] = round(step_bytes / t / 1e6, 1)
            t = timed(nccl_objects, 3)
            comparators["nccl_grouped_send_recv_per_object_GBps_per_rank"] = round(step_bytes / t / 1e6, 1)
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
            comparators["fused_put_kernel_vs_unfused_memcpyPeer_plus_crc32c"] = round(
                kernel_only["put_GBps_per_gpu"] / comparators["unfused_memcpyPeer_plus_crc32c_kernel_GBps_per_rank"], 3)
            comparators["fused_put_kernel_vs_per_object_cudaMemcpyPeerAsync_without_digest"] = round(
                kernel_only["put_GBps_per_gpu"] / comparators["per_object_cudaMemcpyPeerAsync_GBps_per_rank"], 3)

    if dump:
        os.makedirs(args.dump_outputs, exist_ok=True)
        prefix = f"rank{rank}_" if world > 1 else ""
        for name, t in dump.items():
            np.save(os.path.join(args.dump_outputs, prefix + name + ".npy"), t.cpu().numpy())
    cl.stop()
    if world > 1 and cl.dist is not None:
        try:
            cl.dist.destroy_process_group()
        except Exception:
            pass
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        per_gpu = value / world
        if world == 1:
            roof = {"per_gpu_GBps": round(per_gpu, 1), "denominator_GBps": round(peaks.get("hbm_gbs", 6650.0) / 2.0, 1),
                    "denominator": "MEASURED_PEAKS.json hbm_gbs / 2 (every payload byte is read once and written once)"}
            roof["fraction"] = round(per_gpu / roof["denominator_GBps"], 3)
        else:
            measured = comparators.get("cudaMemcpyPeerAsync_single_copy_GBps_per_rank")
            roof = {"per_gpu_GBps": round(per_gpu, 1), "denominator_GBps": NVLINK_NOMINAL_GBPS,
                    "denominator": "NVLink 5 nominal, per direction per GPU (BASELINE.json)",
                    "fraction": round(per_gpu / NVLINK_NOMINAL_GBPS, 3),
                    "measured_peer_copy_peak_GBps": measured,
                    "fraction_of_measured_peer_copy_peak": round(per_gpu / measured, 3) if measured else None,
                    "note": "every payload byte crosses NVLink once per put and once per get; a rank's egress carries its own puts and its neighbour's "
                            "gets.  SM-issued traffic moves in 128-byte packets: pushes top out at ~714 GB/s and bidirectional pulls at ~672 GB/s on "
                            "this fabric whatever the kernel (profiles/r2_nvlink/), copy engines reach ~775 GB/s with larger packets"}
        line = {
            "metric": "batched put+get payload throughput (GB/s), %g MiB random-byte objects, GPU tier, %s fused" % (
                args.object_mib, {"xxh3": "XXH3-64 (per 16 KiB tile) digest", "crc32c": "CRC32C digest", "bbh64": "BBH64 digest", "none": "no digest"}[args.algo]),
            "value": round(value, 2),
            "unit": "GB/s",
            "n_gpus": world,
            "steps": args.steps,
            "warmup": warm,
            "ms_per_step": round(ms / args.steps, 4),
            "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": round(value / BASELINE_GBPS, 1),
            "dtype": "uint8 payload (byte objects; no reduced precision)",
            "data": "synthetic random bytes, device-resident; fresh keys every step; slab recycled by batch_remove",
            "config": {
                "model": "object-store sweep point: batch of %d x %.0f MiB objects per rank" % (nobj, args.object_mib),
                "global_batch": nobj * world,
                "seq_len": osz,
                "parallelism": "ring%d" % world if world > 1 else "local1",
                "placement": "writer's ring neighbour (all payload crosses NVLink)" if world > 1 else "local HBM slab",
                "checksum": args.algo,
                "rank_sync": (args.sync + " (shared-memory rendezvous, host side)") if world > 1 else "n/a",
                "l2_policy": "per-step payload %.2f GiB per rank >> 126 MB L2 (inputs larger than L2)" % (step_bytes / 2**30),
                "control_plane_in_timed_region": "batch_put_start + batch_put_complete + batch_get_workers + batch_remove RPCs every step",
            },
            "kernel_only": kernel_only,
            "kernel_only_by_digest": variants,
            "latency_us_single_object": latency,
            "roofline": roof,
            "e2e": {"value": round(e2e_value, 2), "unit": "GB/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": args.e2e_steps, "ms_per_step": round(e2e_ms / args.e2e_steps, 3),
                    "mode": e2e_mode,
                    "staged_ms_per_step": round(e2e_staged_ms / args.e2e_steps, 3),
                    "zero_copy_ms_per_step": round(e2e_zc_ms / args.e2e_steps, 3),
                    "pipelined_ms_per_step": round(e2e_pipe_ms / args.e2e_steps, 3),
                    "note": "every step: the payload comes from pinned host memory and the WHOLE get result is back in pinned host memory (compared "
                            "byte for byte with the source after the run) -- staged: cudaMemcpyAsync H2D, batch_put_device, batch_get_device, "
                            "cudaMemcpyAsync D2H; zero_copy: batch_put_device is handed the pinned source pointers and batch_get_device the pinned "
                            "destination pointers, the fused kernels move the bytes over PCIe themselves; pipelined: the staged contract with double "
                            "buffers, step i+1's H2D and step i-1's D2H run on copy streams under step i's put / get; value = 2 x payload / time of "
                            "the fastest mode (all reported); PCIe-bound in every mode"},
            "gpu_launches": launches,
            "host_phase_mean_us": phases_max,
            "clocks": clocks,
            "comparators": comparators,
            "baseline_note": "vs_baseline divides by the reference's only throughput figure, an unsourced '~233 MB/sec' config comment (BASELINE.md "
                             "section 1); the reference itself cannot be built or run (see --impl reference)",
        }
        print(json.dumps(line))
    return 0


# ====================================================================================================== other configs
def run_config(args, world: int) -> int:
    import torch

    from blackbird_b200 import _bb
    from blackbird_b200.models import (feature_store_fanout, latency_sweep, replicated_put_verify, throughput_sweep, tier_spill_perf)
    from blackbird_b200.parallel import GpuRankCluster
    from blackbird_b200.utils import ClockSampler

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    sampler = ClockSampler(local_rank, 100).start() if rank == 0 else None
    base = {"n_gpus": world, "higher_is_better": True, "scaling": "weak", "dtype": "uint8 payload", "data": "synthetic random bytes",
            "steps": args.steps, "warmup": max(3, args.warmup)}
    if args.config == "sweep":
        cl = GpuRankCluster(slab_bytes=6 << 30, cluster_id="sweep")
        target = f"gpu{(cl.rank + 1) % cl.world}"
        sizes = [256, 4096, 65536, 1 << 20, 16 << 20] if args.quick else [256, 1024, 4096, 16384, 65536, 262144, 1 << 20, 4 << 20, 16 << 20, 64 << 20, 256 << 20]
        algo = {"xxh3": _bb.ChecksumAlgo.XXH3, "bbh64": _bb.ChecksumAlgo.BBH64, "crc32c": _bb.ChecksumAlgo.CRC32C, "none": _bb.ChecksumAlgo.NONE}[args.algo]
        thr = throughput_sweep(cl, sizes, target, algo=algo)
        lat = latency_sweep(cl, sizes, target, iters=100 if args.quick else 300, algo=algo)
        rows = []
        for t, l in zip(thr, lat):
            row = {"size": t["size"], "batch": t["batch"]}
            for k in ("put_GBps_kernel", "get_GBps_kernel", "put_GBps_client", "get_GBps_client"):
                row[k] = round(cl.sum_over_ranks(t[k]), 2)  # whole job
            for k in ("put_p50_us", "put_p99_us", "get_p50_us", "get_p99_us"):
                row[k] = round(cl.max_over_ranks(l[k]), 1)
            row["rank0_client_phases"] = t.get("phases", {})  # Keystone round trips vs launch vs kernel wait, ms per batch
            rows.append(row)
        cl.stop()
        big = rows[-1]
        line = dict(base, metric="batched put/get GB/s and single-object p50/p99 us vs object size (BASELINE config #2)",
                    value=round(big["put_GBps_client"] + big["get_GBps_client"], 2), unit="GB/s (client-level put + get at the largest size, whole job)",
                    config={"model": "sweep 256 B - 256 MiB, replication 1", "checksum": args.algo, "parallelism": f"ring{world}" if world > 1 else "local1"},
                    sweep=rows)
    elif args.config == "repl3":
        cl = GpuRankCluster(slab_bytes=4 << 30, cluster_id="repl3", nvls_arena_bytes=(256 << 20) if world >= 3 else 0, nvls_group_size=3)
        if world < 3:
            cl.stop()
            line = dict(base, metric="replication=3 batched put (BASELINE config #3)", value=None, unit="GB/s", unavailable="needs >= 3 GPUs")
        else:
            uni = replicated_put_verify(cl, 3, symmetric=False)
            mc = replicated_put_verify(cl, 3, symmetric=True) if cl.arena is not None else None
            agg = lambda r, k: round(cl.sum_over_ranks(r[k]), 1)
            res = {"unicast_fanout": {"put_payload_GBps": agg(uni, "put_payload_GBps"), "put_wire_GBps": agg(uni, "put_wire_GBps"), "get_verified_GBps": agg(uni, "get_GBps")}}
            if mc:
                res["nvls_multicast"] = {"put_payload_GBps": agg(mc, "put_payload_GBps"), "put_delivered_GBps": agg(mc, "put_wire_GBps"),
                                         "get_verified_GBps": agg(mc, "get_GBps"), "multicast_launch_bytes": cl.fabric.path_bytes(True, 3)}
            cl.stop()
            best = max(v["put_payload_GBps"] for v in res.values())
            line = dict(base, metric="replication=3 batched put payload GB/s, CRC32C verified on get from the replicas (BASELINE config #3)", value=best,
                        unit="GB/s (payload, whole job; wire = 3x)", config={"model": "32 x 16 MiB per rank, 3 replicas on distinct GPUs", "parallelism": f"ring{world}"},
                        paths=res)
    elif args.config == "fanout":
        cl = GpuRankCluster(slab_bytes=2 << 30, cluster_id="fanout")
        r1 = feature_store_fanout(cl)
        r3 = feature_store_fanout(cl, replication=3) if world >= 3 else None
        cl.stop()
        line = dict(base, metric="feature-store read fan-out: rank 0 puts 128 x 1 MiB, every rank batch-gets all (BASELINE config #5)",
                    value=round(max(r1["aggregate_get_GBps"], r3["aggregate_get_GBps"] if r3 else 0.0), 1), unit="GB/s (aggregate over readers)",
                    config={"model": "128 x 1 MiB shards", "parallelism": f"1->{world}"}, replication1=r1, replication3=r3)
    else:  # spill
        if world != 1:
            print("bench.py: --config spill runs on one GPU", file=sys.stderr)
            return 2
        import tempfile

        with tempfile.TemporaryDirectory(prefix="bb-nvme-") as nv:
            cl = GpuRankCluster(slab_bytes=(1 << 30) + (64 << 20), cluster_id="spill", dram_bytes=2 << 30, nvme_bytes=6 << 30, nvme_path=nv,
                                high_watermark=0.6, eviction_ratio=0.25)
            res = tier_spill_perf(cl, nobj=48, size=64 << 20)
            cl.stop()
        line = dict(base, metric="GPU->DRAM->NVMe tier spill under memory pressure, 64 MiB objects (BASELINE config #4)", value=res["demotion_GBps"],
                    unit="GB/s (bytes demoted / time spent in the movers)", config={"model": "48 x 64 MiB into a 1 GiB HBM slab, watermark 0.6"}, spill=res)
    clocks = sampler.stop() if sampler else None
    if rank == 0:
        line["clocks"] = clocks
        line["vs_baseline"] = None
        print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
