"""GPU suite (-m gpu), last file on purpose: qualities 2..4 (SURVEY.md 8f rank 1 -- the one-position-per-slot hashers
H2 / H3 / H4 / H54 of c/enc/hash_longest_match_quickly_inc.h, BrotliStoreMetaBlockFast / Trivial of
c/enc/brotli_bit_stream.c:1196-1317) through the C ABI, against digests of the compiled reference, the oracle and the
reference's recorded outputs (brotli_libs.RecordedRef).  Bit-exact.  The device functions of this path are the ones
tests/test_sim.py runs on the CPU (test_sim_q234_*); what only these tests cover is the CUDA plumbing around them: the 32-bit three-pass
radix sort of the slot keys, k_walk<0>, k_verify, k_prep_flat and the host wrapper."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

from brotli_libs import Oracle, RecordedRef
from golden_cases import make_case

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]
HERE = os.path.dirname(__file__)
GOLDEN = json.load(open(os.path.join(HERE, "golden", "golden_oracle_only.json")))
FIXDIR = os.path.join(HERE, "golden", "fixtures")
FIXTURES = json.load(open(os.path.join(HERE, "golden", "fixtures_q234.json")))


@pytest.fixture(scope="module")
def b200():
    import brotli_b200
    assert brotli_b200.available(), "no CUDA device"
    return brotli_b200


def _same(got, want, ctx):
    """Byte equality with a useful failure message (this is the path's first run on hardware)."""
    if got == want:
        return
    if not isinstance(want, bytes):
        raise AssertionError("%r: %d bytes against %r" % (ctx, len(got), want))
    k = next((i for i in range(min(len(got), len(want))) if got[i] != want[i]), min(len(got), len(want)))
    raise AssertionError("%r: %d bytes against %d, first difference at byte %d" % (ctx, len(got), len(want), k))


def test_q234_index_sorted_by_slot(b200):
    """The first thing that differs from the measured path: 32-bit slot keys through three radix passes (k_slot_keys,
    k_radix_*<u32>, k_seg<u32>).  S must be the positions ordered by (slot, position) with the unhashable tail last; seg
    the segment starts.  Checked against numpy (tests/slot_index.py, itself checked against the sim's index on the CPU)
    for H2 / H3 (16 bits), H4 (17 bits) and H54 (20 bits, 7-byte hash)."""
    from corpus import synth_web
    from slot_index import slot_index
    L = b200.lib()
    L.br_debug_sort.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_uint32, C.c_void_p, C.c_void_p]
    for q, n in ((2, 300000), (3, 300000), (4, 300000), (4, 1 << 20), (4, 5000), (2, 9)):
        d = synth_web(n, 17)
        want_S, want_seg, bits = slot_index(d, q)
        S = np.zeros(n, np.uint32); seg = np.zeros((1 << bits) + 2, np.uint32)
        assert L.br_debug_sort(q, 22, d, n, S.ctypes.data, seg.ctypes.data), q
        assert np.array_equal(S, want_S), (q, n, int(np.argmax(S != want_S)))
        assert np.array_equal(seg, want_seg), (q, n)


@pytest.mark.parametrize("g", GOLDEN, ids=lambda g: "%s-%d-q%d-w%d" % (g["kind"], g["n"], g["q"], g["lgwin"]))
def test_q234_golden(b200, g):
    d = make_case(g)
    assert hashlib.sha256(d).hexdigest() == g["in_sha256"]
    out = b200.compress_oneshot(d, g["q"], g["lgwin"])
    assert len(out) == g["out_len"]
    assert hashlib.sha256(out).hexdigest() == g["out_sha256"]


@pytest.mark.parametrize("g", FIXTURES, ids=lambda g: "%s-q%d-w%d" % (g["label"], g["q"], g["lgwin"]))
def test_q234_reference_fixtures(b200, g):
    """The reference's own tests/testdata files at qualities 2..4, against digests of the compiled reference."""
    d = open(os.path.join(FIXDIR, g["file"]), "rb").read()[:g["n"]]
    assert hashlib.sha256(d).hexdigest() == g["in_sha256"]
    out = b200.compress_oneshot(d, g["q"], g["lgwin"])
    assert len(out) == g["out_len"]
    assert hashlib.sha256(out).hexdigest() == g["out_sha256"]


def test_q234_against_oracle_windows(b200):
    ora = Oracle()
    from corpus import synth_binary, synth_text, synth_web
    d1, d2, d3 = synth_text(700000, 31), synth_web(1300000, 32), synth_binary(900000, 34)
    for q in (2, 3, 4):
        for w in (10, 13, 16, 17, 20, 22, 24):
            for d in (d1, d2, d3):
                _same(b200.compress_oneshot(d, q, w), ora.compress(d, q, w), (q, w, len(d)))


def test_q234_edge_sizes(b200):
    ora = Oracle()
    from corpus import synth_text
    base = synth_text(1 << 20, 33) + synth_text(100, 35)
    for n in (1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 63, 64, 65, 511, 512, 4095, 16383, 16384, 16385, 65535, 65536, 65537,
              131072, 131073, (1 << 20) - 1, 1 << 20, (1 << 20) + 1):
        for q in (2, 3, 4):
            _same(b200.compress_oneshot(base[:n], q, 22), ora.compress(base[:n], q, 22), (n, q))
    for d in (bytes(500000), bytes(range(256)) * 3000, b"ab" * 300000, os.urandom(1) * 7 + bytes(70000)):
        for q in (2, 3, 4):
            for w in (12, 22):
                _same(b200.compress_oneshot(d, q, w), ora.compress(d, q, w), (len(d), q, w))


def test_q234_incompressible_and_mixed(b200):
    """Raw metablocks, the sparse-search phases on noise, the late uncompressed fallback (encode.c:604) at quality 2..4."""
    ora = Oracle()
    from corpus import synth_binary, synth_text
    rnd = np.random.default_rng(77).integers(0, 256, 3_000_000, dtype=np.uint8).tobytes()
    mix = synth_text(400000, 78) + rnd[:700000] + synth_binary(500000, 79) + rnd[700000:1000000] + synth_text(300000, 80)
    for q in (2, 3, 4):
        _same(b200.compress_oneshot(rnd, q, 22), ora.compress(rnd, q, 22), q)
        _same(b200.compress_oneshot(mix, q, 20), ora.compress(mix, q, 20), q)


def _drive(b200, d, q, w, sizes, ops):
    c = b200.Compressor(quality=q, lgwin=w)
    out, pos = b"", 0
    for a, op in zip(sizes, ops):
        out += c._stream(d[pos:pos + a], op)
        pos += a
    return out


def test_q234_streaming_flush_and_metadata(b200):
    """PROCESS / FLUSH / EMIT_METADATA / FINISH at quality 2..4 (input blocks of 1 << 14 bytes below quality 4), byte-identical
    to the reference's CompressStream for the same call sequence."""
    from corpus import synth_binary, synth_text
    ref = RecordedRef()
    for d in (synth_text(500000, 61), synth_binary(600000, 62)):
        n = len(d)
        for q, w in ((2, 22), (3, 16), (4, 22), (4, 11)):
            bs = 1 << (14 if q < 4 else 16)
            seqs = [
                ([100000, 50000, 250000, n - 400000], [0, 1, 1, 2]),
                ([0, 300000, 0, n - 300000, 0], [1, 1, 1, 1, 2]),
                ([bs, 0, n - bs], [0, 1, 2]),
                ([4 * bs, 0], [0, 2]),
                ([7, 200000, 5, n - 200012, 0], [3, 0, 3, 1, 2]),
                ([0, 100, 0, 0, 11, n - 111], [3, 1, 3, 1, 3, 2]),
            ]
            for sizes, ops in seqs:
                want = ref.stream_ops(d, q, w, sizes, ops)
                got = _drive(b200, d, q, w, sizes, ops)
                assert got == want, (q, w, sizes, ops, len(got), len(want))


def test_q234_batch_api(b200):
    """BrotliB200CompressBatch at quality 2..4: streams below 1 MiB run as ONE device job per group (k_walk<0, true>: slots,
    windows and the zeroed-table candidate count from each stream's first byte), longer ones one by one; every stream equal
    to the one-shot call."""
    ora = Oracle()
    from corpus import synth_web
    web = synth_web(3_000_000, 90)
    rnd = np.random.default_rng(91)
    streams, off = [], 0
    for i in range(24):
        n = int(rnd.choice([1, 100, 5000, 65536, 200000]))
        streams.append(web[off:off + n]); off += n
    streams.append(web[:1_200_000])          # >= 1 MiB: its own job (H54 at quality 4)
    streams += [b"", bytes(70000), b"ab" * 40000]
    for q, w in ((2, 22), (3, 22), (4, 22), (4, 12), (3, 17)):
        got = b200.compress_batch(streams, q, w)
        assert got == [ora.compress(s, q, w) if s else b"\x06" for s in streams], (q, w)
    many = [web[o:o + 65536] for o in range(0, 2_900_000, 31337)][:600]      # a batch that fills the GPU (2 KiB chunks)
    for q in (2, 4):
        got = b200.compress_batch(many, q, 22)
        assert got == [ora.compress(s, q, 22) for s in many], q


def test_q234_full_size(b200):
    """100 MB of text (BASELINE config C2's input) at quality 2 and 4, and 64 MiB of the binary mix at quality 3 with a 24-bit
    window, against the reference's recorded outputs."""
    from corpus import synth_binary, synth_text
    ref = RecordedRef()
    d = synth_text(100_000_000, 20250922)
    for q in (2, 4):
        _same(b200.compress_oneshot(d, q, 22), ref.compress(d, q, 22), q)
    d = synth_binary(64 << 20, 20250924)
    assert b200.compress_oneshot(d, 3, 24) == ref.compress(d, 3, 24)


def test_q234_fuzz_gpu(b200):
    """Structured random inputs (tests/fuzz_cases.py: periodic data, dictionary words, noise, long runs ...) at quality 2..4
    through the C ABI on the GPU, one-shot and a dozen at a time through the batch call."""
    from brotli_libs import TABLES
    from fuzz_cases import cases, dict_cases
    ora = Oracle()
    todo = [(i, d) for i, d, q, w in cases(31339, 200) if d] + [(1000 + i, d) for i, d, q, w in dict_cases(31340, 40, TABLES) if d]
    for i, d in todo:
        q, w = 2 + i % 3, 10 + (i * 7) % 15
        _same(b200.compress_oneshot(d, q, w), ora.compress(d, q, w), (i, len(d), q, w))
    small = [d for i, d in todo if len(d) < (1 << 20)]
    for a in range(0, len(small), 12):
        part = small[a:a + 12]
        q, w = 2 + (a // 12) % 3, 10 + (a // 12 * 5) % 15
        assert b200.compress_batch(part, q, w) == [ora.compress(x, q, w) for x in part], (a, q, w)


def test_batch_device_resident_quality_2_to_9(b200):
    """BrotliB200CompressBatchDevice at quality 2..9 (added with the quality 2..4 work): streams resident in one device buffer,
    back to back (read in place) and with gaps (gathered on the device), compressed streams packed densely into a device
    buffer; every stream equal to the one-shot call."""
    import torch
    ora = Oracle()
    from corpus import synth_web
    L = b200.lib()
    web = synth_web(2_000_000, 95)
    rnd = np.random.default_rng(96)
    sizes = [int(x) for x in rnd.choice([1, 7, 300, 5000, 65536, 65536, 150000], 40)]
    streams, off = [], 0
    for n in sizes:
        streams.append(web[off:off + n]); off = (off + n) % 1_800_000
    cnt = len(streams)
    for gap in (0, 48):
        offs, o = [], 0
        for x in streams:
            offs.append(o); o += len(x) + gap
        buf = bytearray(o + 64)
        for x, p in zip(streams, offs):
            buf[p:p + len(x)] = x
        d_in = torch.frombuffer(buf, dtype=torch.uint8).cuda()
        cap = sum(len(x) for x in streams) * 2 + 4096 * cnt
        d_out = torch.zeros(cap, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        in_off = (C.c_uint64 * cnt)(*offs)
        in_sz = (C.c_size_t * cnt)(*[len(x) for x in streams])
        for q, w in ((5, 22), (2, 22), (4, 18), (9, 24), (3, 12)):
            out_off = (C.c_uint64 * (cnt + 1))()
            out_sz = (C.c_size_t * cnt)()
            good = L.BrotliB200CompressBatchDevice(q, w, cnt, d_in.data_ptr(), in_off, in_sz, d_out.data_ptr(), cap, out_off, out_sz)
            host = d_out.cpu().numpy().tobytes()
            want = [ora.compress(x, q, w) for x in streams]
            ok = 0
            for k in range(cnt):
                if out_sz[k]:          # (0: above BrotliEncoderMaxCompressedSize, to be sent through the host call)
                    _same(host[out_off[k]:out_off[k] + out_sz[k]], want[k], (gap, q, w, k, len(streams[k])))
                    ok += 1
                else:
                    assert len(want[k]) > L.BrotliEncoderMaxCompressedSize(len(streams[k])), (gap, q, w, k)
            assert good == ok and ok >= cnt - 4, (gap, q, w, good, ok)
            if ok == cnt:
                assert out_off[cnt] == sum(len(x) for x in want)


def test_flush_just_behind_a_block_boundary(b200):
    """All qualities: a FLUSH one or two bytes behind a block boundary leaves a block too short to stitch; the positions the
    block behind it stitches reach back across it (tests/test_sim.py::test_sim_flush_just_behind_a_block_boundary: the case a
    randomized campaign found in the last session, wrong bytes before the fix of br_commit_bits)."""
    from corpus import synth_text
    ref = RecordedRef()
    d = synth_text(300000, 77)
    n = len(d)
    for q, w in ((3, 12), (2, 22), (4, 16), (5, 22), (7, 17), (9, 24)):
        bs = 1 << (14 if q < 4 else 18 if q >= 9 else 16)
        for extra in (1, 2, 3, 6):
            c = bs + extra
            _same(_drive(b200, d, q, w, [c, n - c], [1, 2]), ref.stream_ops(d, q, w, [c, n - c], [1, 2]), (q, w, extra))
        c1, c2 = bs + 1, bs + 2
        _same(_drive(b200, d, q, w, [c1, 1, n - c2], [1, 1, 2]), ref.stream_ops(d, q, w, [c1, 1, n - c2], [1, 1, 2]), (q, w, "two short blocks"))
