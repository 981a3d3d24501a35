"""MXFP8 conformance: every MXFP8 implementation against an exact float64 model of common/mxfp8.h.

The model below is plain numpy and shares no code with the package.  Part one (CPU) checks it against torch's
float8_e4m3fn and then checks the C++ reference (bb.mxfp8_pack_ref / mxfp8_unpack_ref) against it on exhaustive
inputs: every bf16 value as the amax of its block and as an element of blocks 2^1..2^12 times larger, every Inf / NaN
pattern, zero and subnormal blocks, and all 256 x 256 (E4M3 byte, E8M0 byte) pairs.  Part two (gpu) runs the same inputs
through the stand-alone kernels (mxfp8.cu) and the fused transfer kernels (xfer_mxfp8.cu) and requires the same bytes.
"""
import functools

import numpy as np
import pytest
import torch

BLOCK = 32
TILE = 16384  # elements (payload bytes) per fused tile


# ---------------------------------------------------------------------------------------------------------- the model
def _e4m3_values() -> np.ndarray:
    """float64 value of each of the 256 E4M3 codes (S.EEEE.MMM, bias 7); 0x7F / 0xFF are NaN."""
    c = np.arange(256)
    e, m = (c >> 3) & 0xF, c & 7
    mag = np.where(e == 0, m * 2.0 ** -9, (1 + m / 8) * 2.0 ** (e - 7))
    v = np.where(c & 0x80, -mag, mag)
    v[(c & 0x7F) == 0x7F] = np.nan
    return v


E4M3 = _e4m3_values()
E4M3_POS = E4M3[:0x7F]  # finite non-negative codes 0x00..0x7E, increasing
E4M3_MAX = 448.0
NAN_CODE = 0x7F  # every NaN element packs to 0x7F, whatever its sign (common/mxfp8.h)


def model_e4m3(v: np.ndarray) -> np.ndarray:
    """float64 -> E4M3 code: round to nearest, ties to the even code, saturating to +-448, the sign kept (also on 0)."""
    v = np.asarray(v, dtype=np.float64)
    a = np.abs(v)
    fin = np.isfinite(a)
    a_c = np.where(fin, np.minimum(a, E4M3_MAX), E4M3_MAX)
    hi = np.searchsorted(E4M3_POS, a_c, side="left")  # first code whose value >= a
    lo = np.maximum(hi - 1, 0)
    d_lo = a_c - E4M3_POS[lo]
    d_hi = E4M3_POS[np.minimum(hi, 0x7E)] - a_c
    pick_hi = (d_hi < d_lo) | ((d_hi == d_lo) & (hi % 2 == 0))
    code = np.where(pick_hi, hi, lo).astype(np.uint8)
    code = np.where(np.signbit(v), code | 0x80, code).astype(np.uint8)
    return np.where(np.isnan(v), NAN_CODE, code).astype(np.uint8)


def bf16_to_f64(bits: np.ndarray) -> np.ndarray:
    with np.errstate(invalid="ignore"):  # signalling NaNs come out quiet
        return (bits.astype(np.uint32) << 16).view(np.float32).astype(np.float64)


def model_scale(blocks_f64: np.ndarray) -> np.ndarray:
    """E8M0 byte per row of 32 values: floor(log2 amax) - 8 + 127 clamped to [0, 254], amax over the finite |x| (NaN
    skipped); a subnormal amax counts as 2^-127; an all-zero (or all-NaN) block and any block holding an Inf get 127."""
    fin = np.isfinite(blocks_f64)
    amax = np.where(fin, np.abs(blocks_f64), 0.0).max(axis=1)
    has_inf = np.isinf(blocks_f64).any(axis=1)
    _, fe = np.frexp(amax)  # amax = m * 2^fe, m in [0.5, 1)
    exp = np.where(amax < 2.0 ** -126, -127, fe - 1)
    scale = np.clip(exp - 8 + 127, 0, 254)
    return np.where((amax == 0) | has_inf, 127, scale).astype(np.uint8)


def model_pack(bits: np.ndarray):
    """bf16 bit patterns (nblocks, 32) -> (payload (nblocks, 32) uint8, scales (nblocks,) uint8)."""
    f = bf16_to_f64(bits)
    scale = model_scale(f)
    with np.errstate(invalid="ignore"):
        scaled = np.ldexp(f, (127 - scale.astype(np.int64))[:, None])  # exact in float64
    return model_e4m3(scaled), scale


def model_unpack(payload: np.ndarray, scales: np.ndarray):
    """(nblocks, 32) E4M3 codes, (nblocks,) E8M0 bytes -> (bf16 bits, NaN mask).  Byte e decodes to 2^(e-127); 255
    decodes to 2^128, which is +Inf in the float32 the product is formed in.  The product is exact in float64 and its
    float32 rounding is exact unless it overflows; the float32 is rounded to bf16 to nearest even on its bits."""
    s = np.where(scales == 255, np.inf, np.ldexp(1.0, scales.astype(np.int64) - 127))
    with np.errstate(invalid="ignore", over="ignore"):
        prod = E4M3[payload] * s[:, None]
        p32 = prod.astype(np.float32)
    nan = np.isnan(p32)
    u = p32.view(np.uint32).astype(np.uint64)
    bf = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)
    return np.where(nan, 0x7FC0, bf).astype(np.uint16), nan


# --------------------------------------------------------------------------------------------- the exhaustive inputs
def _finite_bf16() -> np.ndarray:
    b = np.arange(1 << 16, dtype=np.uint32)
    return b[(b & 0x7F80) != 0x7F80].astype(np.uint16)  # 65280 patterns, both signs


def _nonfinite_bf16() -> np.ndarray:
    b = np.arange(1 << 16, dtype=np.uint32)
    return b[(b & 0x7F80) == 0x7F80].astype(np.uint16)  # +-Inf and every NaN payload of both signs: 256


def _place(rng, value: np.ndarray, others: np.ndarray) -> np.ndarray:
    """Rows of 32: `others` (n, 31) with `value` (n,) inserted at a position that cycles through 0..31."""
    n = len(value)
    out = np.empty((n, BLOCK), dtype=np.uint16)
    pos = np.arange(n) % BLOCK
    cols = np.arange(BLOCK)[None, :]
    mask = cols == pos[:, None]
    out[mask] = value
    out[~mask] = others.reshape(-1)
    return out


@functools.lru_cache(maxsize=None)
def pack_cases() -> np.ndarray:
    """(nblocks, 32) bf16 bit patterns; an odd block count above 3 Mi elements."""
    rng = np.random.default_rng(20261017)
    fin = _finite_bf16()
    mag = fin & 0x7FFF
    parts = []
    # every finite value sets the amax of its block: the other 31 are random values of no larger magnitude
    others = (rng.integers(0, mag.astype(np.int64)[:, None] + 1, size=(len(fin), BLOCK - 1))
              | (rng.integers(0, 2, size=(len(fin), BLOCK - 1)) << 15)).astype(np.uint16)
    parts.append(_place(rng, fin, others))
    # every finite value in blocks whose amax is 2^k larger (k = 1..12), anchor mantissa 1.0, 1.75 and 1 + 127/128;
    # the 31 values of a block are consecutive in magnitude, the anchor exponent is set from the largest of them
    order = fin[np.lexsort((fin >> 15, mag))]
    pad = (-len(order)) % (BLOCK - 1)
    chunks = np.concatenate([order, order[:pad]]).reshape(-1, BLOCK - 1)
    top_exp = ((chunks & 0x7FFF).max(axis=1) >> 7).astype(np.int64)
    for k in range(1, 13):
        for mant in (0x00, 0x60, 0x7F):
            anchor = (np.minimum(top_exp + k, 254) << 7) | mant | (rng.integers(0, 2, size=len(chunks)) << 15)
            parts.append(_place(rng, anchor.astype(np.uint16), chunks))
    # every Inf / NaN pattern next to finite values: once among values spread over the whole range, once among values
    # small enough that a NaN taken for the amax would change the scale
    nf = _nonfinite_bf16()
    wide = rng.choice(fin, size=(len(nf), BLOCK - 1))
    tiny = (rng.integers(0, 0x0400, size=(len(nf), BLOCK - 1)) | (rng.integers(0, 2, size=(len(nf), BLOCK - 1)) << 15)).astype(np.uint16)
    parts += [_place(rng, nf, wide), _place(rng, nf, tiny)]
    special = [
        np.zeros(BLOCK, np.uint16),                              # all +0
        np.full(BLOCK, 0x8000, np.uint16),                       # all -0
        np.tile(np.array([0x0000, 0x8000], np.uint16), 16),      # +-0 mixed
        np.full(BLOCK, 0x7FC0, np.uint16),                       # all NaN
        np.full(BLOCK, 0xFFC1, np.uint16),                       # all negative NaN
        np.array([0x7F80, 0xFF80] * 16, np.uint16),              # +-Inf only
        np.array([0x7FC0, 0x8000, 0xFF80] + [0x3F80] * 29, np.uint16),  # NaN, -0, -Inf, ones
        np.full(BLOCK, 0x0001, np.uint16),                       # smallest subnormal
        np.full(BLOCK, 0x807F, np.uint16),                       # largest negative subnormal
        np.array([0x7F7F, 0xFF7F] * 16, np.uint16),              # largest finite of both signs
    ]
    parts.append(np.stack(special))
    sub = rng.integers(1, 0x80, size=(64, BLOCK)) | (rng.integers(0, 2, size=(64, BLOCK)) << 15)  # subnormal-only
    parts.append(sub.astype(np.uint16))
    out = np.concatenate(parts)
    if len(out) % 2 == 0:
        out = np.concatenate([out, np.zeros((1, BLOCK), np.uint16)])
    return out


@functools.lru_cache(maxsize=None)
def pair_cases():
    """All 256 x 256 (E4M3 byte, E8M0 byte) pairs: 8 blocks per scale byte, each holding 32 of the 256 codes."""
    payload = np.tile(np.arange(256, dtype=np.uint8).reshape(8, BLOCK), (256, 1))
    scales = np.repeat(np.arange(256, dtype=np.uint8), 8)
    return payload, scales


@functools.lru_cache(maxsize=None)
def packed_model():
    return model_pack(pack_cases())


def packed_bytes(payload: np.ndarray, scales: np.ndarray) -> np.ndarray:
    return np.concatenate([payload.reshape(-1), scales.reshape(-1)])


def assert_bf16_equal(got: np.ndarray, want: np.ndarray, nan: np.ndarray, what: str):
    """Bit-identical, except that any NaN encoding matches a NaN (the sign of zero is compared)."""
    got = got.reshape(-1)
    want = want.reshape(-1)
    nan = nan.reshape(-1)
    got_nan = ((got & 0x7F80) == 0x7F80) & ((got & 0x7F) != 0)
    bad = np.nonzero(np.where(nan, ~got_nan, got != want))[0]
    assert len(bad) == 0, f"{what}: {len(bad)} elements differ, first at {bad[:8].tolist()}: got {[hex(v) for v in got[bad[:8]]]} want {[hex(v) for v in want[bad[:8]]]}"


def assert_bytes_equal(got: np.ndarray, want: np.ndarray, what: str):
    bad = np.nonzero(got.reshape(-1) != want.reshape(-1))[0]
    assert len(bad) == 0, f"{what}: {len(bad)} bytes differ, first at {bad[:8].tolist()}: got {got.reshape(-1)[bad[:8]].tolist()} want {want.reshape(-1)[bad[:8]].tolist()}"


# ------------------------------------------------------------------------------------------------- part one: CPU only
def test_model_e4m3_rounding_matches_torch_float8():
    bf = bf16_to_f64(_finite_bf16())
    mids = (E4M3_POS[1:] + E4M3_POS[:-1]) / 2  # every tie between neighbouring codes, and one float32 ulp either side
    m32 = mids.astype(np.float32)
    near = np.concatenate([m32, np.nextafter(m32, np.float32(0)), np.nextafter(m32, np.float32(np.inf))]).astype(np.float64)
    v = np.concatenate([bf, near, -near, E4M3_POS, -E4M3_POS, [448.0, 463.99, 464.0, -464.0]])
    ref = torch.from_numpy(v.astype(np.float32)).to(torch.float8_e4m3fn).view(torch.uint8).numpy()
    defined = (ref & 0x7F) != 0x7F  # torch turns |x| past the saturation point into NaN; the model saturates
    assert defined.sum() > 30000
    assert_bytes_equal(model_e4m3(v[defined]), ref[defined], "model vs torch float8_e4m3fn")
    assert (model_e4m3(np.array([1e6, -1e6, np.inf, -np.inf, 500.0])) == [0x7E, 0xFE, 0x7E, 0xFE, 0x7E]).all()
    # the decode table is torch's, too
    codes = np.arange(256, dtype=np.uint8)
    tv = torch.from_numpy(codes).view(torch.float8_e4m3fn).double().numpy()
    assert np.array_equal(np.isnan(tv), np.isnan(E4M3))
    fin = ~np.isnan(E4M3)
    assert np.array_equal(tv[fin], E4M3[fin]) and np.array_equal(np.signbit(tv[fin]), np.signbit(E4M3[fin]))


def test_pack_cases_cover_the_edges():
    cases = pack_cases()
    n = cases.size
    assert n > 3 * 2 ** 20 and (n // BLOCK) % 2 == 1
    payload, scales = packed_model()
    assert set(np.unique(scales)) == set(range(0, 247))  # every reachable scale byte, including the clamp to 0
    f = bf16_to_f64(cases)
    assert (np.isnan(f).sum(axis=1) > 0).sum() >= 256 and (np.isinf(f).sum(axis=1) > 0).sum() >= 2
    fin = np.isfinite(f)
    amax_mant = np.frexp(np.where(fin, np.abs(f), 0).max(axis=1))[0] * 2
    assert (amax_mant >= 1.75).sum() > 10000  # blocks whose largest element saturates to 448
    assert ((payload & 0x7F) == 0x7E)[fin].sum() > 10000
    assert ((payload == 0x80) & fin).sum() > 1000  # -0, and negatives that round to zero
    assert set(cases.reshape(-1).tolist()) == set(range(1 << 16))  # every bf16 bit pattern


def test_cpu_pack_matches_model(bb):
    cases = pack_cases()
    payload, scales = packed_model()
    got = np.frombuffer(bb.mxfp8_pack_ref(cases.reshape(-1)), dtype=np.uint8)
    n = cases.size
    assert_bytes_equal(got[n:], scales, "CPU reference scales")
    assert_bytes_equal(got[:n], payload, "CPU reference payload")


def test_cpu_unpack_matches_model_on_every_pair(bb):
    payload, scales = pair_cases()
    want, nan = model_unpack(payload, scales)
    got = np.frombuffer(bb.mxfp8_unpack_ref(packed_bytes(payload, scales), payload.size), dtype=np.uint16)
    assert_bf16_equal(got, want, nan, "CPU reference unpack")


def test_scale_zero_round_trip(bb):
    """A block whose amax is below 2^-118 gets scale byte 0, which decodes to 2^-127 (not to zero)."""
    x = np.arange(0x0100, 0x0120, dtype=np.uint16)  # ~2^-125
    payload, scales = model_pack(x.reshape(1, BLOCK))
    assert scales[0] == 0 and (payload != 0).all()
    back, _ = model_unpack(payload, scales)
    assert (back != 0).all() and (np.abs(bf16_to_f64(back) - bf16_to_f64(x)) <= bf16_to_f64(x) * 2 ** -3).all()
    got = np.frombuffer(bb.mxfp8_unpack_ref(packed_bytes(payload, scales), BLOCK), dtype=np.uint16)
    assert np.array_equal(got, back.reshape(-1))


# ------------------------------------------------------------------------------------------------------ part two: GPU
GUARD = 64  # bytes of sentinel before and after every region a kernel writes


def _cuda_or_fail():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need CUDA (marked gpu)")
    return torch.cuda.current_stream().cuda_stream


def _up(a: np.ndarray) -> torch.Tensor:
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()


class Guarded:
    """Regions at 16-byte aligned offsets of one device buffer, each between GUARD bytes of a sentinel."""

    def __init__(self, sizes, sentinel: int):
        self.offs = []
        off = GUARD
        for s in sizes:
            self.offs.append(off)
            off += (s + GUARD + 15) // 16 * 16
        self.sizes = list(sizes)
        self.sentinel = sentinel
        self.buf = torch.full((off,), sentinel, dtype=torch.uint8, device="cuda")

    def ptr(self, i) -> int:
        return self.buf.data_ptr() + self.offs[i]

    def host(self) -> np.ndarray:
        return self.buf.cpu().numpy()

    def region(self, h: np.ndarray, i) -> np.ndarray:
        return h[self.offs[i]:self.offs[i] + self.sizes[i]]

    def check_guards(self, h: np.ndarray, what: str):
        outside = np.ones(len(h), dtype=bool)
        for o, s in zip(self.offs, self.sizes):
            outside[o:o + s] = False
        bad = np.nonzero(outside & (h != self.sentinel))[0]
        assert len(bad) == 0, f"{what}: {len(bad)} guard bytes overwritten, first at {bad[:8].tolist()}"


def _unpack_stream():
    """Packed input of the unpack tests: the model-packed pack cases followed by all (E4M3, E8M0) pairs."""
    p0, s0 = packed_model()
    p1, s1 = pair_cases()
    return np.concatenate([p0, p1]), np.concatenate([s0, s1])


@pytest.mark.gpu
def test_gpu_standalone_pack_matches_model(bb):
    s = _cuda_or_fail()
    cases = pack_cases()
    n = cases.size
    payload, scales = packed_model()
    src = _up(cases)
    g = Guarded([n + n // BLOCK], 0xA5)
    bb.mxfp8_pack(src.data_ptr(), n, g.ptr(0), s)
    torch.cuda.synchronize()
    h = g.host()
    g.check_guards(h, "mxfp8_pack")
    got = g.region(h, 0)
    assert_bytes_equal(got[n:], scales, "mxfp8_pack scales")
    assert_bytes_equal(got[:n], payload, "mxfp8_pack payload")


@pytest.mark.gpu
def test_gpu_standalone_unpack_matches_model(bb):
    s = _cuda_or_fail()
    payload, scales = _unpack_stream()
    n = payload.size
    want, nan = model_unpack(payload, scales)
    src = _up(packed_bytes(payload, scales))
    g = Guarded([2 * n], 0xA5)
    bb.mxfp8_unpack(src.data_ptr(), n, g.ptr(0), s)
    torch.cuda.synchronize()
    h = g.host()
    g.check_guards(h, "mxfp8_unpack")
    assert_bf16_equal(g.region(h, 0).view(np.uint16), want, nan, "mxfp8_unpack")
    # scale byte 0 on its own: not flushed to zero
    zero = scales == 0
    assert (want.reshape(-1, BLOCK)[zero] != 0).any()


# Object sizes of one fused batch (elements): a tail-only object, objects either side of one tile, one with three tiles
# and a tail, a 64-tile object and a run of 1-tile objects -- 40 in all.  The input stream is cut into such batches.
LAYOUT = [32, TILE - 32, TILE, TILE + 32, 3 * TILE + 7 * 32, 64 * TILE] + [TILE] * 34


def _batches(total: int):
    """[[(first element, n_elems), ...], ...] covering [0, total) with LAYOUT, the last batch cut short."""
    out, pos = [], 0
    while pos < total:
        batch = []
        for sz in LAYOUT:
            if pos >= total:
                break
            sz = min(sz, total - pos)
            batch.append((pos, sz))
            pos += sz
        out.append(batch)
    return out


def _obj_packed(payload: np.ndarray, scales: np.ndarray, a: int, n: int) -> np.ndarray:
    return np.concatenate([payload.reshape(-1)[a:a + n], scales.reshape(-1)[a // BLOCK:(a + n) // BLOCK]])


MAX_CTAS = [1, 2, 5, 0]  # 0: the launch default (one CTA per SM, at most 128)


@pytest.mark.gpu
@pytest.mark.parametrize("max_ctas", MAX_CTAS)
def test_gpu_fused_pack_matches_model(bb, max_ctas):
    """bb_xfer_fp8 put: 1-3 replicas per object, every replica byte-identical to the model, guards intact, digest =
    BBH64 of the model's packed object."""
    s = _cuda_or_fail()
    cases = pack_cases()
    payload, scales = packed_model()
    src = _up(cases)
    eng = bb.XferEngine(0, 1024, 2)
    eng.set_max_ctas(max_ctas)
    sentinel = 0xA5 if MAX_CTAS.index(max_ctas) % 2 == 0 else 0x5A
    for batch in _batches(cases.size):
        nrep = [1 + i % 3 for i in range(len(batch))]
        sizes = [n + n // BLOCK for (_, n), r in zip(batch, nrep) for _ in range(r)]
        g = Guarded(sizes, sentinel)
        items, k = [], 0
        for (a, n), r in zip(batch, nrep):
            items.append((src.data_ptr() + 2 * a, [g.ptr(k + j) for j in range(r)], n))
            k += r
        dg, st, _ = eng.run_fp8(items, False, s)
        torch.cuda.synchronize()
        assert st == [0] * len(batch)
        h = g.host()
        g.check_guards(h, f"fused pack, max_ctas {max_ctas}")
        k = 0
        for i, ((a, n), r) in enumerate(zip(batch, nrep)):
            want = _obj_packed(payload, scales, a, n)
            for j in range(r):
                assert_bytes_equal(g.region(h, k + j), want, f"fused pack object {i} ({n} elements) replica {j}, max_ctas {max_ctas}")
            assert dg[i] == bb.bbh64(want), f"digest of object {i} ({n} elements), max_ctas {max_ctas}"
            k += r


@pytest.mark.gpu
@pytest.mark.parametrize("max_ctas", MAX_CTAS)
def test_gpu_fused_unpack_matches_model(bb, max_ctas):
    """bb_xfer_fp8 get: bf16 output bit-identical to the model (NaN as a class), guards intact, verified digests give a
    zero status; one flipped payload byte and one flipped scale byte flag exactly those two objects."""
    s = _cuda_or_fail()
    payload, scales = _unpack_stream()
    want, nan = model_unpack(payload, scales)
    want, nan = want.reshape(-1), nan.reshape(-1)
    eng = bb.XferEngine(0, 1024, 2)
    eng.set_max_ctas(max_ctas)
    sentinel = 0xA5 if MAX_CTAS.index(max_ctas) % 2 == 0 else 0x5A
    for bi, batch in enumerate(_batches(payload.size)):
        objs = [_obj_packed(payload, scales, a, n) for a, n in batch]
        slab = Guarded([len(o) for o in objs], 0)
        hs = np.zeros(slab.buf.numel(), dtype=np.uint8)
        for i, o in enumerate(objs):
            hs[slab.offs[i]:slab.offs[i] + len(o)] = o
        slab.buf.copy_(torch.from_numpy(hs))
        digests = [bb.bbh64(o) for o in objs]
        out = Guarded([2 * n for _, n in batch], sentinel)
        items = [(out.ptr(i), slab.ptr(i), n, d) for i, ((_, n), d) in enumerate(zip(batch, digests))]
        dg, st, _ = eng.run_fp8(items, True, s)
        torch.cuda.synchronize()
        assert st == [0] * len(batch) and dg == digests
        h = out.host()
        out.check_guards(h, f"fused unpack, max_ctas {max_ctas}")
        for i, (a, n) in enumerate(batch):
            assert_bf16_equal(out.region(h, i).view(np.uint16), want[a:a + n], nan[a:a + n],
                              f"fused unpack object {i} ({n} elements), max_ctas {max_ctas}")
        if bi == 0:
            p_obj, s_obj = 5, 3  # 64-tile object: a payload byte; 16384 + 32 object: a byte of its scales
            slab.buf[slab.offs[p_obj] + 12345] ^= 0x10
            slab.buf[slab.offs[s_obj] + batch[s_obj][1] + 7] ^= 0x01
            _, st, _ = eng.run_fp8(items, True, s)
            torch.cuda.synchronize()
            assert st == [1 if i in (p_obj, s_obj) else 0 for i in range(len(batch))]
