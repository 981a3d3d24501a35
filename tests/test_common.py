"""common/: error model, json-lite, yaml-lite, checksums (CPU golden models)."""
import os

import numpy as np
import pytest

REFERENCE_CONFIGS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_configs")


def test_error_codes_domains_and_strings(bb):
    E = bb.ErrorCode
    # numeric parity with the reference's 1000-spaced domains (error_domain.h:14-38)
    assert int(E.OK) == 0 and int(E.INTERNAL_ERROR) == 1000 and int(E.BUFFER_OVERFLOW) == 2000
    assert int(E.NETWORK_ERROR) == 3000 and int(E.ETCD_ERROR) == 4000 and int(E.OBJECT_NOT_FOUND) == 5000
    assert int(E.CLIENT_ERROR) == 6000 and int(E.CONFIG_ERROR) == 7000
    assert int(E.NOT_IMPLEMENTED) == 1005 and int(E.INSUFFICIENT_SPACE) == 2006 and int(E.CHECKSUM_MISMATCH) == 5007
    assert bb.error_domain(E.CHECKSUM_MISMATCH) == "DATA" and bb.error_domain(E.OK) == "SUCCESS"
    # every code has a name and a description (the reference misses NOT_IMPLEMENTED / INSUFFICIENT_SPACE)
    for name, code in E.__members__.items():
        assert bb.error_string(code) == name
        assert bb.error_description(code) not in ("", "Unknown error code")


def test_json_roundtrip_and_errors(bb):
    s = '{"a":[1,2.5,true,null,"x\\n\\u00e9"],"b":{"c":-7,"big":18446744073709551615}}'
    v = bb.parse_json(s)
    assert v["a"][0] == 1 and v["a"][1] == 2.5 and v["a"][2] is True and v["a"][3] is None and v["a"][4] == "x\n\u00e9"
    assert v["b"]["c"] == -7
    assert bb.parse_json(bb.json_roundtrip(s)) == v
    for bad in ['{"a":}', '[1,2', '{"a":1} x', '"unterminated', '{"a" 1}']:
        with pytest.raises(ValueError):
            bb.parse_json(bad)


def test_yaml_reference_configs(bb):
    ks = bb.parse_yaml(open(os.path.join(REFERENCE_CONFIGS, "keystone.yaml")).read())
    assert ks["keystone"]["cluster_id"] == "blackbird_cluster"
    assert ks["keystone"]["etcd_endpoints"] == ["localhost:2379"]
    assert ks["keystone"]["high_watermark"] == 0.8 and ks["keystone"]["enable_ha"] is False
    assert ks["logging"]["level"] == "INFO"
    w = bb.parse_yaml(open(os.path.join(REFERENCE_CONFIGS, "worker.yaml")).read())
    assert w["worker"]["interconnects"] == ["rdma", "tcp"]
    assert w["storage_pools"][0] == {"pool_id": "ram_pool_0", "storage_class": "RAM_CPU", "size_bytes": 2147483648}
    cxl = bb.parse_yaml(open(os.path.join(REFERENCE_CONFIGS, "cxl_worker.yaml")).read())
    pools = cxl["worker"]["storage_pools"]
    assert pools[1]["config"]["dax_device"] == "/dev/dax0.0" and pools[1]["capacity"] == "256_GB"
    assert cxl["worker"]["allocation"]["preferred_tiers"][3]["max_size"] == "unlimited"


def test_yaml_subset_features(bb):
    doc = """
# comment
a: 1
b:
  - x
  - k: v   # inline map item
    z: [1, 2, "three"]
  - {p: 1, q: two}
c: "quoted: colon"
d: 'it''s'
e: ~
f: 0x10
"""
    v = bb.parse_yaml(doc)
    assert v == {"a": 1, "b": ["x", {"k": "v", "z": [1, 2, "three"]}, {"p": 1, "q": "two"}], "c": "quoted: colon",
                 "d": "it's", "e": None, "f": 16}
    with pytest.raises(ValueError):
        bb.parse_yaml("a:\n\t- tab")
    assert bb.parse_size("32_GB") == 32 << 30 and bb.parse_size("10 MiB") == 10 << 20 and bb.parse_size("4k") == 4096
    assert bb.parse_size("2147483648") == 2147483648 and bb.parse_size("bogus") is None


def test_crc32c_golden_and_algebra(bb):
    assert bb.crc32c(b"123456789") == 0xE3069283  # iSCSI check value
    assert bb.crc32c(b"") == 0
    assert bb.crc32c(bytes(32)) == 0x8A9136AA
    assert bb.crc32c(bytes([0xFF] * 32)) == 0x62A8AB43
    a, b = os.urandom(100003), os.urandom(77771)
    assert bb.crc32c(a) == bb.crc32c_sw(a)
    assert bb.crc32c(b, bb.crc32c(a)) == bb.crc32c(a + b)  # chaining
    assert bb.crc32c_combine(bb.crc32c(a), bb.crc32c(b), len(b)) == bb.crc32c(a + b)
    ra, rb = bb.crc32c_raw(a), bb.crc32c_raw(b)
    assert bb.crc32c_raw(a + b) == bb.gf2_mulmod(ra, bb.gf2_xpow_bytes(len(b))) ^ rb
    assert bb.crc32c_raw(bytes(37) + a) == ra  # leading zeros do not change a raw remainder
    assert bb.crc32c_from_raw(ra, len(a)) == bb.crc32c(a)
    assert bb.gf2_mulmod(0x80000000, 0x12345678) == 0x12345678  # 0x80000000 is the polynomial "1"


def _bbh64_numpy(bb, x):
    n = len(x)
    T = 16384
    mask = (1 << 64) - 1

    def sm(v):
        v = (v + 0x9E3779B97F4A7C15) & mask
        v = ((v ^ (v >> 30)) * 0xBF58476D1CE4E5B9) & mask
        v = ((v ^ (v >> 27)) * 0x94D049BB133111EB) & mask
        return v ^ (v >> 31)

    def mix(v):
        v ^= v >> 33
        v = (v * 0xFF51AFD7ED558CCD) & mask
        v ^= v >> 33
        v = (v * 0xC4CEB9FE1A85EC53) & mask
        return v ^ (v >> 33)

    W = np.array([[bb.bbh64_weight(k, c) for c in range(16)] for k in range(128)], dtype=np.uint64)
    KN = [sm(c + 1) | 1 for c in range(16)]
    o = np.arange(T)
    rows, ks = (o >> 10) * 8 + ((o & 127) >> 4), (((o & 1023) >> 7) << 4) + (o & 15)
    s = 0
    for t in range((n + T - 1) // T):
        tile = np.zeros(T, dtype=np.uint64)
        chunk = x[t * T:(t + 1) * T]
        tile[:len(chunk)] = chunk
        A = np.zeros((128, 128), dtype=np.uint64)
        A[rows, ks] = tile
        D = A @ W
        for m in range(128):
            r = sum(int(D[m, c]) * KN[c] for c in range(16)) & mask
            s = (s + mix((r + (t * 128 + m + 1) * 0x9E3779B97F4A7C15) & mask)) & mask
    return mix(s ^ ((n * 0xD6E8FEB86659FD93) & mask))


def test_bbh64_matches_independent_numpy_model(bb):
    rng = np.random.default_rng(7)
    for n in [0, 1, 16, 4096, 16384, 16385, 50001]:
        x = rng.integers(0, 256, size=n, dtype=np.uint8)
        assert bb.bbh64(x) == _bbh64_numpy(bb, x), n


def test_bbh64_detects_changes(bb):
    rng = np.random.default_rng(3)
    x = rng.integers(0, 256, size=70000, dtype=np.uint8)
    h = bb.bbh64(x)
    y = x.copy()
    y[12345] ^= 1
    assert bb.bbh64(y) != h  # single bit flip
    z = x.copy()
    z[100], z[101] = x[101], x[100]
    assert bb.bbh64(z) != h or x[100] == x[101]  # transposition
    t = x.copy()
    t[:16384], t[16384:32768] = x[16384:32768].copy(), x[:16384].copy()
    assert bb.bbh64(t) != h  # whole-tile swap (position dependence)
    assert bb.bbh64(np.concatenate([x, np.zeros(1, np.uint8)])) != h  # length extension with zeros
    # layout bijection of the UMMA canonical tile
    seen = {(bb.bbh64_off_to_row(o), bb.bbh64_off_to_k(o)) for o in range(16384)}
    assert len(seen) == 16384 and all(0 <= m < 128 and 0 <= k < 128 for m, k in seen)


def test_bbh64_simd_paths_match_the_byte_at_a_time_definition(bb):
    """bbh64() dispatches to AVX-512 VNNI / AVX2 code on the host tiers and TCP clients; every path computes the same
    integers as the reference definition (which the CUDA kernels are tested against), tile sums add up across ranges."""
    import numpy as np

    rng = np.random.default_rng(5)
    assert bb.bbh64_impl_name() in ("avx512-vnni", "avx2", "scalar")
    for n in (0, 1, 15, 16, 4095, 16384, 16385, 100_000, (1 << 20) + 7):
        a = rng.integers(0, 256, n, dtype=np.uint8)
        ref = bb.bbh64_reference(a)
        assert bb.bbh64(a) == ref
        for impl in ("scalar", "avx2", "avx512-vnni"):
            got = bb.bbh64_using(impl, a)
            assert got is None or got == ref, (impl, n)
    for v in (255, 128, 1):  # accumulator extremes: 128 x 255 x 255 per column must not wrap or saturate
        a = np.full(3 * 16384 + 100, v, dtype=np.uint8)
        assert bb.bbh64(a) == bb.bbh64_reference(a)
        assert bb.bbh64_using("avx2", a) in (None, bb.bbh64_reference(a))
    a = rng.integers(0, 256, (5 << 20) + 123, dtype=np.uint8)
    tiles = (a.size + 16383) // 16384
    parts = [bb.bbh64_partial(a, 0, 100), bb.bbh64_partial(a, 100, 57), bb.bbh64_partial(a, 157, tiles - 157)]
    assert bb.bbh64_finalize(sum(parts) & ((1 << 64) - 1), a.size) == bb.bbh64(a)


def test_json_surrogate_escapes(bb):
    """\\uXXXX pairs decode to one code point; a surrogate that is not part of a pair becomes U+FFFD instead of an invalid
    code point (found by review of a -Wmaybe-uninitialized warning; Python's own encoder never emits such input)."""
    assert bb.parse_json('"\\ud83d\\ude00"') == "\U0001F600"
    assert bb.parse_json('"\\ud83d\\u0041"') == "\ufffdA" and bb.parse_json('"\\ud83dA"') == "\ufffdA"
    assert bb.parse_json('"\\ude00x"') == "\ufffdx" and bb.parse_json('"\\ud83d"') == "\ufffd"


def test_sha256_and_hmac_match_hashlib(bb):
    """The handshake's SHA-256 / HMAC-SHA256 against hashlib, across every padding boundary and long keys."""
    import hashlib
    import hmac
    import os
    assert bb.sha256(b"abc").hex() == "ba7816bf8f01cfea414140de5dae2223b00361a396177a9cb410ff61f20015ad"
    for n in list(range(0, 130)) + [191, 192, 255, 256, 1000, 4096, 100_003]:
        data = os.urandom(n)
        assert bb.sha256(data) == hashlib.sha256(data).digest(), n
    for klen in (0, 1, 20, 63, 64, 65, 200):
        key = os.urandom(klen)
        for n in (0, 1, 55, 56, 64, 300):
            msg = os.urandom(n)
            assert bb.hmac_sha256(key, msg) == hmac.new(key, msg, hashlib.sha256).digest(), (klen, n)


def test_xxh3_tiles_are_the_standard_xxh3_64_and_the_combine_matches_the_model(bb):
    """ChecksumAlgo.XXH3 (csrc/common/xxh3.h): every 16 KiB tile is hashed with the unmodified XXH3-64 (checked against the
    python-xxhash binding of the reference implementation), tiles are combined by the position-keyed commutative sum."""
    import os

    xxhash = pytest.importorskip("xxhash")
    for _ in range(8):
        t = os.urandom(16384)
        assert bb.xxh3_tile(t) == xxhash.xxh3_64_intdigest(t)
    assert bb.xxh3_tile(bytes(16384)) == xxhash.xxh3_64_intdigest(bytes(16384))
    M = (1 << 64) - 1
    GOLD, LENMUL = 0x9E3779B97F4A7C15, 0xD6E8FEB86659FD93

    def mix64(x):
        x ^= x >> 33
        x = (x * 0xff51afd7ed558ccd) & M
        x ^= x >> 33
        x = (x * 0xc4ceb9fe1a85ec53) & M
        return x ^ (x >> 33)

    def model(b):
        s = 0
        for t in range((len(b) + 16383) // 16384):
            tile = b[t * 16384:(t + 1) * 16384].ljust(16384, b"\0")
            s = (s + mix64((xxhash.xxh3_64_intdigest(tile) + (t + 1) * GOLD) & M)) & M
        return mix64(s ^ ((len(b) * LENMUL) & M))

    for n in [0, 1, 100, 4096, 16383, 16384, 16385, 100000, (1 << 20) + 7]:
        b = os.urandom(n)
        assert bb.xxh3t64(b) == model(b), n
    # slices add up (what parallel streams / chunked hashing / GPU RAW_SUM slices rely on)
    b = os.urandom(5 * 16384 + 100)
    parts = (bb.xxh3t64_partial(b, 0, 2) + bb.xxh3t64_partial(b, 2, 3) + bb.xxh3t64_partial(b, 5, 1)) & M
    assert bb.bbh64_finalize(parts, len(b)) == bb.xxh3t64(b)
    # position dependence and length binding
    assert bb.xxh3t64(b[16384:] + b[:16384]) != bb.xxh3t64(b) and bb.xxh3t64(b + b"\0") != bb.xxh3t64(b)
