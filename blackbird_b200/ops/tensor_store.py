"""Torch-facing API: put / get CUDA tensors through the object store with the fused kernels.

    store = TensorStore(cluster.client)
    store.batch_put(["act/0", "act/1"], [t0, t1])                  # BBH64 digest fused into the copy
    store.put("kv/layer3", kv_bf16, pack_fp8=True)                  # block-scaled MXFP8 on the wire / in the slab
    t = store.get("kv/layer3")                                      # verified + unpacked bf16 tensor

Tensor metadata (dtype, shape, packing) travels in a small side object `<key>#meta`.
"""
from __future__ import annotations

import json
from typing import Optional, Sequence

import torch

from .. import _bb

_DTYPES = {str(d).replace("torch.", ""): d for d in (torch.uint8, torch.int8, torch.int16, torch.int32, torch.int64, torch.float16,
                                                     torch.bfloat16, torch.float32, torch.float64, torch.bool)}


class TensorStore:
    def __init__(self, client, config: Optional["_bb.WorkerConfig"] = None):
        self.client = client
        self.config = config or _bb.WorkerConfig(replication_factor=1, max_workers_per_copy=1,
                                                 preferred_classes=[_bb.StorageClass.RAM_GPU])

    @staticmethod
    def _stream() -> int:
        return torch.cuda.current_stream().cuda_stream

    def _meta_cfg(self):
        return _bb.WorkerConfig(replication_factor=self.config.replication_factor, max_workers_per_copy=1, ttl_ms=self.config.ttl_ms,
                                enable_soft_pin=self.config.enable_soft_pin, checksum=_bb.ChecksumAlgo.CRC32C)

    # ------------------------------------------------------------------ put
    def _fused_fp8_ok(self, t: torch.Tensor, cfg) -> bool:
        """Pack fused into the put kernel: bf16, a whole number of 32-element MX blocks, up to 3 copies (one tile pass
        fans out to every replica), each copy in one shard."""
        return (t.dtype == torch.bfloat16 and self.client.device_fp8_eligible(t.numel()) and 1 <= cfg.replication_factor <= 3
                and cfg.max_workers_per_copy == 1 and t.data_ptr() % 16 == 0)

    def batch_put(self, keys: Sequence[str], tensors: Sequence[torch.Tensor], pack_fp8: bool = False, config=None) -> None:
        cfg = config or self.config
        keys = list(keys)
        tensors = [t.contiguous() for t in tensors]
        if pack_fp8:
            # objects the fused kernel can take go through batch_put_device_fp8 (bf16 read once, packed bytes on the
            # wire, digest of the packed object from the tensor cores); the rest are packed first (unfused path below)
            fused = [i for i, t in enumerate(tensors) if t.is_cuda and self._fused_fp8_ok(t, cfg)]
            if fused:
                fk = [keys[i] for i in fused]
                ecs = self.client.batch_put_device_fp8(fk, [tensors[i].data_ptr() for i in fused], [tensors[i].numel() for i in fused],
                                                       cfg, self._stream())
                done = [i for i, e in zip(fused, ecs) if e == _bb.ErrorCode.OK]
                bad = [(keys[i], e) for i, e in zip(fused, ecs) if e not in (_bb.ErrorCode.OK, _bb.ErrorCode.NOT_IMPLEMENTED)]
                if bad:
                    raise RuntimeError(f"fused fp8 put failed: {bad[:3]}")
                metas = []
                for i in done:
                    t = tensors[i]
                    metas.append(json.dumps({"dtype": "bfloat16", "shape": list(t.shape), "packed": "mxfp8", "numel": t.numel(),
                                             "padded_numel": t.numel()}).encode())
                if done:
                    ecs = self.client.batch_put([keys[i] + "#meta" for i in done], metas, self._meta_cfg())
                    if any(e != _bb.ErrorCode.OK for e in ecs):
                        raise RuntimeError("meta put failed")
                rest = [i for i in range(len(keys)) if i not in set(done)]
                keys, tensors = [keys[i] for i in rest], [tensors[i] for i in rest]
                if not keys:
                    return
        payloads, metas, keep = [], [], []
        for t in tensors:
            assert t.is_cuda, "TensorStore moves CUDA tensors (host data: use client.put)"
            meta = {"dtype": str(t.dtype).replace("torch.", ""), "shape": list(t.shape), "packed": None, "numel": t.numel()}
            if pack_fp8:
                assert t.dtype == torch.bfloat16, "MXFP8 packing takes bf16 tensors"
                n = t.numel()
                npad = (n + 31) // 32 * 32
                src = t.view(-1)
                if npad != n:
                    src = torch.cat([src, torch.zeros(npad - n, dtype=t.dtype, device=t.device)])
                packed = torch.empty(_bb.mxfp8_packed_bytes(npad), dtype=torch.uint8, device=t.device)
                _bb.mxfp8_pack(src.data_ptr(), npad, packed.data_ptr(), self._stream())
                keep.append(src)
                meta["packed"] = "mxfp8"
                meta["padded_numel"] = npad
                t = packed
            assert t.data_ptr() % 16 == 0, "tensor storage must be 16-byte aligned"
            payloads.append(t)
            metas.append(json.dumps(meta).encode())
        ecs = self.client.batch_put_device(list(keys), [p.data_ptr() for p in payloads], [p.numel() * p.element_size() for p in payloads],
                                           cfg, self._stream())
        bad = [(k, e) for k, e in zip(keys, ecs) if e != _bb.ErrorCode.OK]
        if bad:
            raise RuntimeError(f"put failed: {bad[:3]}")
        ecs = self.client.batch_put([k + "#meta" for k in keys], metas, self._meta_cfg())
        if any(e != _bb.ErrorCode.OK for e in ecs):
            raise RuntimeError("meta put failed")

    def put(self, key: str, tensor: torch.Tensor, pack_fp8: bool = False, config=None) -> None:
        self.batch_put([key], [tensor], pack_fp8, config)

    # ------------------------------------------------------------------ get
    def batch_get(self, keys: Sequence[str], device: Optional[torch.device] = None) -> list:
        device = device or torch.device("cuda", torch.cuda.current_device())
        metas = []
        for ec, blob in self.client.batch_get([k + "#meta" for k in keys]):
            if ec != _bb.ErrorCode.OK:
                raise KeyError(f"object metadata missing: {ec}")
            metas.append(json.loads(blob))
        keys = list(keys)
        result = [None] * len(keys)
        # MXFP8 objects made of whole tiles: unpack fused into the get kernel (falls through when the object is not a
        # single GPU-fabric shard any more, e.g. after demotion to a host tier)
        fused = [i for i, m in enumerate(metas) if m["packed"] == "mxfp8" and m["padded_numel"] == m["numel"]
                 and self.client.device_fp8_eligible(m["numel"])]
        if fused:
            outs = [torch.empty(metas[i]["numel"], dtype=torch.bfloat16, device=device) for i in fused]
            ecs = self.client.batch_get_device_fp8([keys[i] for i in fused], [o.data_ptr() for o in outs], [metas[i]["numel"] for i in fused],
                                                   self._stream())
            for i, o, e in zip(fused, outs, ecs):
                if e == _bb.ErrorCode.OK:
                    result[i] = o.view(metas[i]["shape"])
                elif e != _bb.ErrorCode.NOT_IMPLEMENTED:
                    raise RuntimeError(f"fused fp8 get failed: {keys[i]}: {e}")
        rest = [i for i in range(len(keys)) if result[i] is None]
        if not rest:
            return result
        all_keys, all_metas = keys, metas
        keys, metas = [all_keys[i] for i in rest], [all_metas[i] for i in rest]
        bufs = []
        for m in metas:
            if m["packed"] == "mxfp8":
                bufs.append(torch.empty(_bb.mxfp8_packed_bytes(m["padded_numel"]), dtype=torch.uint8, device=device))
            else:
                bufs.append(torch.empty(m["shape"], dtype=_DTYPES[m["dtype"]], device=device))
        ecs, sizes = self.client.batch_get_device(list(keys), [b.data_ptr() for b in bufs], [b.numel() * b.element_size() for b in bufs],
                                                  self._stream())
        bad = [(k, e) for k, e in zip(keys, ecs) if e != _bb.ErrorCode.OK]
        if bad:
            raise RuntimeError(f"get failed: {bad[:3]}")
        out = []
        for m, b in zip(metas, bufs):
            if m["packed"] == "mxfp8":
                t = torch.empty(m["padded_numel"], dtype=torch.bfloat16, device=device)
                _bb.mxfp8_unpack(b.data_ptr(), m["padded_numel"], t.data_ptr(), self._stream())
                out.append(t[: m["numel"]].view(m["shape"]))
            else:
                out.append(b)
        for i, t in zip(rest, out):
            result[i] = t
        return result

    def get(self, key: str, device: Optional[torch.device] = None) -> torch.Tensor:
        return self.batch_get([key], device)[0]

    # ------------------------------------------------------------------ paged KV blocks
    @staticmethod
    def _block_segments(caches: Sequence[torch.Tensor], block_ids: Sequence[torch.Tensor]):
        """(S, 2) int64 segment table (pointer, bytes) and per-object segment counts: object i is, cache by cache in list
        order, caches[c][block_ids[i][j]] for every j."""
        if not caches:
            raise ValueError("batch_*_blocks needs at least one cache tensor")
        bases, strides, lens, nblocks = [], [], [], []
        for c in caches:
            if not c.is_cuda:
                raise ValueError("caches must be CUDA tensors")
            if c.dim() < 1 or c.shape[0] == 0:
                raise ValueError(f"a cache is [num_blocks, ...]; got shape {tuple(c.shape)}")
            if not c[0].is_contiguous():
                raise ValueError(f"each cache must be contiguous in its trailing dimensions (shape {tuple(c.shape)}, stride {c.stride()})")
            es = c.element_size()
            block = c[0].numel() * es
            if c.data_ptr() % 16 or (c.stride(0) * es) % 16 or block % 16:
                raise ValueError(f"cache blocks must start 16-byte aligned and be a multiple of 16 bytes (block {block} B, "
                                 f"stride {c.stride(0) * es} B, base {c.data_ptr():#x})")
            bases.append(c.data_ptr())
            strides.append(c.stride(0) * es)
            lens.append(block)
            nblocks.append(c.shape[0])
        bases = torch.tensor(bases, dtype=torch.int64)[:, None]
        strides = torch.tensor(strides, dtype=torch.int64)[:, None]
        lens = torch.tensor(lens, dtype=torch.int64)[:, None]
        limit = min(nblocks)
        rows, counts = [], []
        for ids in block_ids:
            ids = torch.as_tensor(ids).to("cpu", torch.int64).reshape(-1)
            if ids.numel() == 0:
                raise ValueError("every key needs at least one block")
            if int(ids.min()) < 0 or int(ids.max()) >= limit:
                raise IndexError(f"block index out of range [0, {limit})")
            ptr = bases + ids[None, :] * strides                      # [cache, block]
            rows.append(torch.stack([ptr.reshape(-1), lens.expand(-1, ids.numel()).reshape(-1)], 1))
            counts.append(ptr.numel())
        return torch.cat(rows), counts

    def batch_put_blocks(self, keys: Sequence[str], caches: Sequence[torch.Tensor], block_ids: Sequence[torch.Tensor], config=None) -> None:
        """Stores object keys[i] = the blocks block_ids[i] of every cache (cache by cache, in list order) with one fused
        gather put: no staging copy.  The object is the same as a contiguous put of those blocks concatenated, so
        `get` returns it as a flat uint8 tensor and `remove` / `keys` work on it."""
        keys = list(keys)
        if len(keys) != len(block_ids):
            raise ValueError("one block list per key")
        cfg = config or self.config
        segs, counts = self._block_segments(caches, block_ids)
        ecs = self.client.batch_put_device_gather(keys, segs, counts, cfg, self._stream())
        bad = [(k, e) for k, e in zip(keys, ecs) if e != _bb.ErrorCode.OK]
        if bad:
            raise RuntimeError(f"block put failed: {bad[:3]}")
        sizes, pos = [], 0
        for n in counts:
            sizes.append(int(segs[pos:pos + n, 1].sum()))
            pos += n
        metas = [json.dumps({"dtype": "uint8", "shape": [s], "packed": None, "numel": s}).encode() for s in sizes]
        ecs = self.client.batch_put([k + "#meta" for k in keys], metas, self._meta_cfg())
        if any(e != _bb.ErrorCode.OK for e in ecs):
            raise RuntimeError("meta put failed")

    def batch_get_blocks(self, keys: Sequence[str], caches: Sequence[torch.Tensor], block_ids: Sequence[torch.Tensor]) -> None:
        """Writes object keys[i] into the blocks block_ids[i] of every cache (the layout of batch_put_blocks; the block
        ids may differ from the ones it was stored from) with one fused scatter get.  The blocks must add up to the
        stored size.  Block lists that overlap receive unspecified bytes."""
        keys = list(keys)
        if len(keys) != len(block_ids):
            raise ValueError("one block list per key")
        segs, counts = self._block_segments(caches, block_ids)
        ecs = self.client.batch_get_device_scatter(keys, segs, counts, self._stream())
        bad = [(k, e) for k, e in zip(keys, ecs) if e != _bb.ErrorCode.OK]
        if bad:
            raise RuntimeError(f"block get failed: {bad[:3]}")

    def remove(self, keys: Sequence[str]) -> None:
        self.client.batch_remove(list(keys) + [k + "#meta" for k in keys])

    def keys(self, prefix: str = "", limit: int = 0) -> list:
        """Names of the tensors stored under `prefix` (key order; the `#meta` side objects are hidden)."""
        out, after = [], ""
        while True:
            page = self.client.keystone().list_objects(prefix, 1000, after)
            out += [k for k, _, _, _ in page if not k.endswith("#meta")]
            if len(page) < 1000 or (limit and len(out) >= limit):
                return out[:limit] if limit else out
            after = page[-1][0]


class AsyncTensorStore(TensorStore):
    """TensorStore whose puts / gets run on a side stream from a worker thread, so they overlap the caller's compute
    (KV-cache offload, activation checkpoints).  `put_async` orders itself after the work already queued on the
    caller's stream (event wait), returns a `concurrent.futures.Future`; `get_async`'s future yields the tensors, already
    synchronised with the side stream.  The native calls release the GIL."""

    def __init__(self, client, config=None, workers: int = 1):
        super().__init__(client, config)
        from concurrent.futures import ThreadPoolExecutor

        self._pool = ThreadPoolExecutor(max_workers=workers, thread_name_prefix="bb-async")
        self._device = torch.cuda.current_device()
        self._side = torch.cuda.Stream(device=self._device)

    def _stream(self) -> int:  # every native call of this store is issued on the side stream
        return self._side.cuda_stream

    def put_async(self, keys: Sequence[str], tensors: Sequence[torch.Tensor], pack_fp8: bool = False, config=None):
        ready = torch.cuda.Event()
        ready.record(torch.cuda.current_stream())  # the tensors' producers
        tensors = list(tensors)  # keep them alive until the transfer is done

        def run():
            torch.cuda.set_device(self._device)
            self._side.wait_event(ready)
            with torch.cuda.stream(self._side):
                self.batch_put(keys, tensors, pack_fp8, config)
            self._side.synchronize()
            return len(tensors)

        return self._pool.submit(run)

    def get_async(self, keys: Sequence[str]):
        def run():
            torch.cuda.set_device(self._device)
            with torch.cuda.stream(self._side):
                out = self.batch_get(keys)
            self._side.synchronize()
            return out

        return self._pool.submit(run)

    def put_blocks_async(self, keys: Sequence[str], caches: Sequence[torch.Tensor], block_ids: Sequence[torch.Tensor], config=None):
        ready = torch.cuda.Event()
        ready.record(torch.cuda.current_stream())  # the blocks' producers
        caches, block_ids = list(caches), list(block_ids)

        def run():
            torch.cuda.set_device(self._device)
            self._side.wait_event(ready)
            with torch.cuda.stream(self._side):
                self.batch_put_blocks(keys, caches, block_ids, config)
            self._side.synchronize()
            return len(keys)

        return self._pool.submit(run)

    def get_blocks_async(self, keys: Sequence[str], caches: Sequence[torch.Tensor], block_ids: Sequence[torch.Tensor]):
        ready = torch.cuda.Event()
        ready.record(torch.cuda.current_stream())  # work queued on the destination blocks so far
        caches, block_ids = list(caches), list(block_ids)

        def run():
            torch.cuda.set_device(self._device)
            self._side.wait_event(ready)
            with torch.cuda.stream(self._side):
                self.batch_get_blocks(keys, caches, block_ids)
            self._side.synchronize()
            return len(keys)

        return self._pool.submit(run)

    def close(self):
        self._pool.shutdown(wait=True)
