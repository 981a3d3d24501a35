"""Multi-GPU data-plane correctness (SURVEY §4: "GPU data-plane correctness (bit-exact + CRC) at 1/2/4/8 GPUs").
Runs tests/multi_gpu_worker.py under torchrun on min(#GPUs, 4) ranks; skipped on a single-GPU box."""
import json
import os
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _json_objects(text):
    dec, out, i = json.JSONDecoder(), [], 0
    while True:
        i = text.find('{"rank"', i)
        if i < 0:
            return out
        try:
            obj, end = dec.raw_decode(text, i)
            out.append(obj)
            i = end
        except ValueError:
            i += 1


def test_ring_replication_fanout_and_remote_dram_on_n_gpus():
    import torch

    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    world = min(n, 4)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "multi_gpu_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    lines = _json_objects(r.stdout)  # ranks print concurrently: two objects may share a line
    assert len(lines) == world and all(x["ring"] == "ok" and "remote_dram_pool" in x for x in lines), lines
