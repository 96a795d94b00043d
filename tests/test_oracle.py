"""CPU suite, part 1: the oracle (oracle/brotli_oracle.c) against the golden vectors made from the
compiled reference, and against the reference's recorded outputs (brotli_libs.RecordedRef)."""
import hashlib
import json
import os

import pytest

from brotli_libs import PRODUCT_SO, Oracle, RecordedRef
from golden_cases import make_case

GOLDEN = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden.json")))
GOLDEN_ORACLE_ONLY = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden_oracle_only.json")))
FAST = [g for g in GOLDEN if g["n"] <= 2_500_000] + GOLDEN_ORACLE_ONLY


FIXDIR = os.path.join(os.path.dirname(__file__), "golden", "fixtures")
FIXTURES = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "fixtures.json")))


def fixture_bytes(g):
    """The reference's own test files (byte copies under tests/golden/fixtures, see make_fixture_golden.py)."""
    d = open(os.path.join(FIXDIR, g["file"]), "rb").read()
    return d[:g["n"]]


@pytest.fixture(scope="module")
def oracle():
    return Oracle()


@pytest.mark.parametrize("g", FIXTURES, ids=lambda g: "%s-q%d-w%d" % (g["label"], g["q"], g["lgwin"]))
def test_oracle_on_reference_fixtures(oracle, g):
    """The oracle on the reference's tests/testdata files, against digests of the compiled reference; includes
    BASELINE.json config C1 = alice29.txt[:65536] at quality 5, lgwin 22 (24 091 bytes)."""
    d = fixture_bytes(g)
    assert hashlib.sha256(d).hexdigest() == g["in_sha256"]
    out = oracle.compress(d, g["q"], g["lgwin"])
    assert len(out) == g["out_len"] and hashlib.sha256(out).hexdigest() == g["out_sha256"]


@pytest.mark.parametrize("g", FAST, ids=lambda g: "%s-%d-q%d-w%d" % (g["kind"], g["n"], g["q"], g["lgwin"]))
def test_oracle_matches_golden(oracle, g):
    d = make_case(g)
    assert hashlib.sha256(d).hexdigest() == g["in_sha256"], "corpus generator drifted"
    out = oracle.compress(d, g["q"], g["lgwin"])
    assert len(out) == g["out_len"]
    assert hashlib.sha256(out).hexdigest() == g["out_sha256"]


def test_oracle_matches_reference_and_roundtrips(oracle):
    ref = RecordedRef()
    for g in FAST[:12]:
        d = make_case(g)
        a = ref.compress(d, g["q"], g["lgwin"])
        assert a == oracle.compress(d, g["q"], g["lgwin"])
        assert ref.decompress(a, len(d)) == d


def test_empty_input_and_bounds():
    """The reference's output for empty input, and its BrotliEncoderMaxCompressedSize, which the product's must equal."""
    import ctypes as C
    ref = RecordedRef()
    assert ref.compress(b"", 5, 22) == b"\x06"
    lib = C.CDLL(PRODUCT_SO, mode=os.RTLD_LOCAL)      # built by build(); its host-only entry points need no GPU
    lib.BrotliEncoderMaxCompressedSize.restype = C.c_size_t
    lib.BrotliEncoderMaxCompressedSize.argtypes = [C.c_size_t]
    for n in (0, 1, 100, 1 << 14, (1 << 24) + 5):
        assert ref.max_compressed_size(n) >= n
        assert lib.BrotliEncoderMaxCompressedSize(n) == ref.max_compressed_size(n), n


def test_fast_log2_table(oracle):
    # c/enc/fast_log.c:13: the table literals carry an 'f' suffix -> float-rounded values
    import math
    import struct
    for v in (1, 2, 3, 7, 100, 255):
        f = struct.unpack("f", struct.pack("f", math.log2(v)))[0]
        assert oracle.lib.oracle_fast_log2(v) == f
    assert oracle.lib.oracle_fast_log2(4096) == 12.0


def test_q1_oracle_against_reference(oracle):
    """Quality 1 (compress_fragment_two_pass.c): one-shot calls over every table size / min_match the
    reference can pick, and the streaming call pattern of c/tools/brotli.c (512 KiB PROCESS calls)."""
    from corpus import synth_binary, synth_text, synth_web
    ref = RecordedRef()
    base = synth_web(3_000_000, 51)
    for n in (0, 1, 15, 16, 17, 255, 256, 257, 1000, 5000, 40000, 65536, 131072, 131073, 300000, 1 << 20, 3_000_000):
        for w in (10, 16, 18, 22, 24):
            assert oracle.compress(base[:n], 1, w) == ref.compress(base[:n], 1, w), (n, w)
    for d in (synth_text(1_400_000, 52), synth_binary(1_400_000, 53), bytes(300000)):
        for w in (17, 22):
            assert oracle.compress(d, 1, w) == ref.compress(d, 1, w)
    chunk = 1 << 19
    for n in (0, 100, chunk, chunk + 1, 3 * chunk, 3_000_000):
        d = base[:n]
        calls = [min(chunk, n - o) for o in range(0, n, chunk)]
        if n % chunk == 0:
            calls.append(0)
        for w in (16, 22):
            assert oracle.compress_q1_stream(d, w, calls) == ref.compress_stream(d, 1, w, chunk), (n, w)


def test_q234_oracle_against_reference(oracle):
    """Qualities 2..4 (H2 / H3 / H4 / H54, fast / trivial / context-free meta-blocks): oracle groundwork for
    SURVEY.md 8f rank 1, pinned against the reference over window sizes and hasher switches."""
    from corpus import synth_binary, synth_web
    ref = RecordedRef()
    base = synth_web(2_200_000, 71)
    for n in (0, 1, 7, 8, 9, 100, 5000, 16384, 16385, 70000, 300000, (1 << 20) - 1, 1 << 20, 2_200_000):
        for q in (2, 3, 4):
            for w in (10, 16, 17, 22):
                assert oracle.compress(base[:n], q, w) == ref.compress(base[:n], q, w), (n, q, w)
    d = synth_binary(1_300_000, 72)
    for q in (2, 3, 4):
        assert oracle.compress(d, q, 24) == ref.compress(d, q, 24)
