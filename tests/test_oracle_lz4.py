"""CPU: pins oracle/lz4_ref.c against the real upstream codec (liblz4, what CodecLz4 wraps) and the compression ratios
printed in the reference's docs/src/index.md:52-63.  What upstream produced for the inputs below is stored in
tests/golden/lz4_upstream.json (written by tests/golden/make_golden.py with the system liblz4 1.9.4), so the comparison needs
no liblz4 at test time."""
import hashlib
import json
import os

import numpy as np
import pytest


@pytest.fixture(scope="module")
def upstream():
    return json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "lz4_upstream.json")))


def _sha(b):
    return hashlib.sha256(b).hexdigest()


def _bodies(oracle):
    rng = np.random.default_rng(11)
    N = 65536
    brands = ["apple", "samsung", "huawai", "microsoft", "dell", "xbox", "sony", "intel"]
    return {
        "id": np.arange(1, N + 1, dtype=np.int64).tobytes(),
        "rand1000": rng.integers(1, 1001, N).astype(np.int64).tobytes(),
        "brands": oracle.block_body("String", [brands[i] for i in rng.integers(0, 8, N)], 0, N),
        "price": (1 + 0.1 * rng.integers(0, 19991, N)).astype(np.float64).tobytes(),
        "f01": rng.random(N).tobytes(),
        "zeros": bytes(70000),
        "tiny": b"abc",
        "twelve": b"abcabcabcabc",
        "thirteen": b"aaaaaaaaaaaaa",
        "mixed": bytes(300) + rng.integers(0, 256, 999).astype(np.uint8).tobytes() + b"xyz" * 1000,
    }


def corrupt_streams(oracle):
    """(body, good stream, damaged streams): 300 damaged copies of one compressed block, every third one also truncated."""
    rng = np.random.default_rng(5)
    body = rng.integers(1, 50, 5000).astype(np.int64).tobytes()
    good = oracle.compress_block(body)
    streams = []
    for trial in range(300):
        bad = bytearray(good)
        k = int(rng.integers(0, len(bad)))
        bad[k] ^= int(rng.integers(1, 256))
        if trial % 3 == 0:
            bad = bad[: int(rng.integers(1, len(bad)))]
        streams.append(bytes(bad))
    return body, good, streams


def test_documented_compression_ratios(oracle):
    """docs/src/index.md:52-63: id 2.0, rand(1:1000) 2.55, 8 brands 2.85, rand(1.:0.1:2000.) 1.93 (accel 2, 65536-row blocks)."""
    b = _bodies(oracle)
    for name, want in [("id", 2.0), ("rand1000", 2.55), ("brands", 2.85), ("price", 1.93)]:
        for comp in (oracle.lz4_compress(b[name], 2), oracle.compress_block(b[name])):
            assert abs(len(b[name]) / len(comp) - want) < 0.02, (name, len(b[name]) / len(comp))


def test_round_trip_both_directions_with_upstream_liblz4(oracle, upstream):
    """The restated compressor emits upstream's LZ4_compress_fast stream byte for byte (so upstream's decoder reads it), and
    the restated decoder reads it back."""
    bodies = _bodies(oracle)
    assert sorted(bodies) == sorted(upstream["compress"])
    for name, body in bodies.items():
        exp = upstream["compress"][name]
        assert _sha(body) == exp["body_sha256"], f"{name}: the input is not the one upstream compressed"
        for accel in (1, 2, 8):
            own = oracle.lz4_compress(body, accel)
            up = exp["accel"][str(accel)]
            assert len(own) == up["size"] and _sha(own) == up["sha256"], (name, accel)    # same greedy parse as LZ4_compress_fast
            assert oracle.lz4_decompress(own, len(body)) == body, name


def test_corrupt_streams_are_rejected_like_upstream(oracle, upstream):
    """LZ4_decompress_safe's verdict on every damaged stream (accepted: sha256 of what it wrote; refused: null)."""
    body, good, streams = corrupt_streams(oracle)
    exp = upstream["corrupt"]
    assert _sha(good) == exp["good_sha256"] and len(streams) == len(exp["verdicts"])
    disagreements = 0
    for bad, want in zip(streams, exp["verdicts"]):
        try:
            got = _sha(oracle.lz4_decompress(bad, len(body)))
        except oracle.OracleError:
            got = None
        if (got is None) != (want is None):
            disagreements += 1
        elif got is not None:
            assert got == want
    assert disagreements == 0


def test_block_stream_framing(oracle):
    """test/block_streams.jl:11-67: one compressed block of 64000 Int64 in 1..100000 reads back equal; a second
    block of another size follows a skipped first one."""
    import struct
    rng = np.random.default_rng(1)
    a = rng.integers(1, 100001, 64000).astype(np.int64)
    b = rng.integers(1, 100001, 74000).astype(np.int64)
    frames = []
    for arr in (a, b):
        body = arr.tobytes()
        comp = oracle.compress_block(body)
        frames.append(struct.pack("<iqq", len(arr), len(body), len(comp)) + comp)
    rows, body = oracle.decode_block(frames[0], a.nbytes)
    assert rows == 64000 and np.array_equal(np.frombuffer(body, np.int64), a)
    # skip_block: header + compressed bytes, then the next block decodes
    stream = frames[0] + frames[1]
    r0, _, c0 = struct.unpack("<iqq", stream[:20])
    assert r0 == 64000
    rows, body = oracle.decode_block(stream[20 + c0:], b.nbytes)
    assert rows == 74000 and np.array_equal(np.frombuffer(body, np.int64), b)
