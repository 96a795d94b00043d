"""CPU suite, part 2: the product's warp-task device code (LZ77 walkers, chain, entropy coder)
compiled for the host by tests/sim/br_sim.cc with a one-lane warp, against the oracle.  This is
how the bit-exact logic is debugged without a GPU; the CUDA build itself is checked by -m gpu."""
import ctypes as C
import os

import numpy as np
import pytest

from brotli_libs import ROOT, TABLES, Oracle
from golden_cases import CASES, make_case

SIM_SO = os.path.join(ROOT, "tests", "sim", "libbrsim.so")


@pytest.fixture(scope="module")
def sim():
    if not os.path.exists(SIM_SO):
        import __graft_entry__
        __graft_entry__.build_checkers()
    L = C.CDLL(SIM_SO)
    L.sim_init.argtypes = [C.c_char_p, C.c_size_t, C.c_uint32]
    L.sim_compress.restype = C.c_long
    L.sim_compress.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_uint32, C.c_void_p, C.c_size_t, C.c_void_p]
    blob = open(TABLES, "rb").read()
    L.sim_init(blob, len(blob), (1 << 22) + 2)
    L.sim_q1_compress.restype = C.c_long
    L.sim_q1_compress.argtypes = [C.c_int, C.c_char_p, C.c_uint32, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
    L.sim_q1_compress_seg.restype = C.c_long
    L.sim_q1_compress_seg.argtypes = [C.c_int, C.c_char_p, C.c_uint32, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                      C.c_int, C.c_int, C.c_uint32, C.c_void_p]
    return L


SMALL = [c for c in CASES if c["n"] <= 1_500_000 and not (c["kind"] in ("binary", "heavy") and c["q"] == 9)]


@pytest.mark.parametrize("c", SMALL, ids=lambda c: "%s-%d-q%d-w%d" % (c["kind"], c["n"], c["q"], c["lgwin"]))
def test_sim_matches_oracle(sim, c):
    d = make_case(c)
    if c["q"] == 1:
        # quality 1: the stream as the device code makes it (the one-shot wrapper's empty-input and
        # raw-stream rules live in br_api.cc)
        want = Oracle().compress_q1_stream(d, c["lgwin"])
        cap = 2 * len(d) + 100000
        out = C.create_string_buffer(cap)
        r = sim.sim_q1_compress(c["lgwin"], d, len(d), None, 0, out, cap)
        assert r >= 0 and out.raw[:r] == want
        return
    want = Oracle().compress(d, c["q"], c["lgwin"])
    cap = len(d) + len(d) // 2 + 4096
    out = C.create_string_buffer(cap)
    st = np.zeros(8, np.uint32)
    r = sim.sim_compress(c["q"], c["lgwin"], d, len(d), out, cap, st.ctypes.data)
    assert r >= 0
    assert out.raw[:r] == want


def test_sim_q1_call_patterns(sim):
    """Quality 1 cuts fragments per CompressStream call (encode.c:1425): the device code planned with
    the same call sizes gives the oracle's stream."""
    from corpus import synth_web
    d = synth_web(700000, 41)
    ora = Oracle()
    for calls in ([700000], [524288, 175712], [100000] * 7 + [0], [1, 15, 16, 17, 699951], [0, 700000, 0]):
        for w in (12, 18, 22):
            want = ora.compress_q1_stream(d, w, calls)
            arr = (C.c_size_t * len(calls))(*calls)
            cap = 2 * len(d) + 100000
            out = C.create_string_buffer(cap)
            r = sim.sim_q1_compress(w, d, len(d), arr, len(calls), out, cap)
            assert r >= 0 and out.raw[:r] == want, (calls, w)


def test_sim_q1_flush_segments(sim):
    """FLUSH at quality 1: the stream is a chain of byte-aligned segments (window bits only in the first,
    byte padding behind every flushed one): device code per segment == oracle for the whole op sequence."""
    from corpus import synth_web
    d = synth_web(500000, 42)
    ora = Oracle()
    cases = [([0, 500000], [1, 2]), ([100000, 0, 400000, 0], [1, 1, 1, 2]), ([1, 2, 3, 499994], [1, 1, 0, 2]),
             ([200000, 150000, 150000], [0, 1, 2]), ([250000, 250000, 0], [1, 1, 2])]
    for sizes, ops in cases:
        for w in (16, 22):
            want = ora.compress_q1_stream(d, w, sizes, ops)
            got, pos, seg_calls, seg_start, header = b"", 0, [], 0, 1
            for a, op in zip(sizes, ops):
                if a or op == 2:
                    seg_calls.append(a)
                pos += a
                if op in (1, 2):
                    piece = d[seg_start:pos]
                    if op == 2 and not header and not piece:
                        got += b"\x03"
                    elif piece or header:
                        arr = (C.c_size_t * max(1, len(seg_calls)))(*seg_calls)
                        cap = 2 * len(piece) + 100000
                        out = C.create_string_buffer(cap)
                        r = sim.sim_q1_compress_seg(w, piece, len(piece), arr if seg_calls else None, len(seg_calls), out, cap, header, op, 0, None)
                        assert r >= 0
                        got += out.raw[:r]
                        header = 0
                    seg_calls, seg_start = [], pos
            assert got == want, (sizes, ops, w)


def test_sim_q1_segments_mid_byte(sim):
    """Bounded-memory streaming at quality 1: the stream is cut into device segments between calls; a segment that
    neither flushes nor finishes ends mid-byte and the next one starts behind its pending bits (encode.c:1445
    last_bytes_).  Device code per segment, stitched the way br_api.cc q1_segment does == oracle for the op sequence."""
    from corpus import synth_web
    d = synth_web(400000, 7) + bytes(np.random.default_rng(5).integers(0, 256, 70000, dtype=np.uint8))
    ora = Oracle()
    cases = [([100000, 200000, 170000], [0, 0, 2]), ([1, 65536, 70000, 334463], [0, 0, 1, 2]),
             ([300000, 100000, 70000, 0], [0, 0, 0, 2]), ([131072, 131072, 207856], [0, 1, 2]), ([470000], [2])]
    for sizes, ops in cases:
        for w in (16, 18, 22):
            want = ora.compress_q1_stream(d, w, sizes, ops)
            got, pos, header, bits, byte = bytearray(), 0, 1, 0, 0
            for a, op in zip(sizes, ops):
                piece = d[pos:pos + a]
                pos += a
                if not piece:
                    assert op == 2 and not header
                    acc = (byte & ((1 << bits) - 1)) | (3 << bits)
                    got += acc.to_bytes((bits + 2 + 7) // 8, "little")
                    continue
                arr = (C.c_size_t * 1)(a)
                cap = 2 * a + 100000
                out = C.create_string_buffer(cap)
                eb = C.c_uint32(0)
                r = sim.sim_q1_compress_seg(w, piece, a, arr, 1, out, cap, header, op, bits, C.byref(eb))
                assert r >= 0 and (eb.value + 7) // 8 == r
                seg = bytearray(out.raw[:r])
                if bits:
                    assert seg[0] & ((1 << bits) - 1) == 0
                    seg[0] |= byte & ((1 << bits) - 1)
                bits, byte, header = 0, 0, 0
                if op == 0 and eb.value & 7:
                    bits, byte = eb.value & 7, seg.pop()
                got += seg
            assert bytes(got) == want, (sizes, ops, w)


def _fuzz_check(sim, d, q, w):
    ora = Oracle()
    cap = 2 * len(d) + 100000
    out = C.create_string_buffer(cap)
    if q == 1:
        r = sim.sim_q1_compress(w, d, len(d), None, 0, out, cap)
        return r >= 0 and out.raw[:r] == ora.compress_q1_stream(d, w)
    if not d:
        return True
    st = np.zeros(8, np.uint32)
    r = sim.sim_compress(q, w, d, len(d), out, cap, st.ctypes.data)
    return r >= 0 and out.raw[:r] == ora.compress(d, q, w)


def test_sim_fuzz_regressions(sim):
    """Inputs found by fuzzing that broke the speculative parse (see tests/fuzz_cases.py)."""
    from fuzz_cases import REGRESSIONS, cases
    by_seed = {}
    for seed, idx in REGRESSIONS:
        by_seed.setdefault(seed, set()).add(idx)
    for seed, idxs in by_seed.items():
        for i, d, q, w in cases(seed, max(idxs) + 1):
            if i in idxs:
                assert _fuzz_check(sim, d, q, w), (seed, i, len(d), q, w)


def test_sim_fuzz_sample(sim):
    from fuzz_cases import cases, dict_cases
    for i, d, q, w in cases(20250922, 120):
        if len(d) <= 120000:
            assert _fuzz_check(sim, d, q, w), (i, len(d), q, w)
    for i, d, q, w in dict_cases(20250923, 40, TABLES):
        assert _fuzz_check(sim, d, q, w), ("dict", i, len(d), q, w)


def _sim_cuts(sim, d, q, w, hint, cuts, kinds, is_final, finish_empty=0, lgblock=0, disable_ctx=0, stream_offset=0, with_header=1):
    sim.sim_compress_cuts.restype = C.c_long
    sim.sim_compress_cuts.argtypes = [C.c_int, C.c_int, C.c_uint32, C.c_char_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32,
                                      C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_uint32]
    cp = (C.c_uint32 * max(1, len(cuts)))(*cuts)
    ck = (C.c_uint32 * max(1, len(cuts)))(*kinds)
    eb = (C.c_uint64 * max(1, len(cuts)))()
    cap = len(d) + len(d) // 2 + 4096
    out = C.create_string_buffer(cap)
    st = np.zeros(8, np.uint32)
    r = sim.sim_compress_cuts(q, w, hint, d, len(d), cp, ck, len(cuts), is_final, with_header, finish_empty, eb, out, cap, st.ctypes.data,
                              lgblock, disable_ctx, stream_offset)
    assert r >= 0
    return out.raw[:r]


def test_sim_flush_cuts_and_parameters(sim):
    """The device code with the input cut by FLUSH operations (encode.c:1356, :1700), with FINISH arriving without input
    behind a full block (encode.c:520), and with BROTLI_PARAM_LGBLOCK / DISABLE_LITERAL_CONTEXT_MODELING, against the
    reference's CompressStream driven with the same calls (recorded: brotli_libs.RecordedRef)."""
    from brotli_libs import RecordedRef
    from corpus import synth_binary, synth_text, synth_web
    ref = RecordedRef()
    for d in (synth_text(400000, 3), synth_binary(600000, 5)):
        n = len(d)
        for q, w in ((5, 22), (9, 24), (7, 19)):
            bs = 1 << (18 if (q >= 9 and w >= 18) else 16)
            for sizes, ops in (([100000, 50000, n - 150000], [0, 1, 2]), ([bs, 0, n - bs, 0], [0, 1, 1, 2]), ([100, n - 100, 0], [1, 0, 2])):
                want = ref.stream_ops(d, q, w, sizes, ops)
                pos, cuts, acc, fixed, hint = 0, [], 0, False, 0
                for a, op in zip(sizes, ops):
                    if not fixed and (op != 0 or acc + a >= bs):   # encode.c:1619: the size hint freezes at the first EncodeData
                        hint, fixed = acc + a, True
                    acc += a
                    pos += a
                    if op == 1 and pos > 0 and (not cuts or cuts[-1] != pos):
                        cuts.append(pos)
                if cuts and cuts[-1] == n:
                    got = _sim_cuts(sim, d, q, w, hint, cuts, [1] * len(cuts), 0) + b"\x03"
                else:
                    got = _sim_cuts(sim, d, q, w, hint, cuts, [1] * len(cuts), 1)
                assert got == want, (q, w, sizes, ops)
    # quality 7..9 above 1 MiB: the pilot launch (BrParams::pilot) with the input cut by FLUSH, incl. a first block of 2 bytes
    d = synth_web(1_400_000, 3)
    for q, w in ((9, 24), (7, 18)):
        for sizes, ops in (([500000, 0, 900000, 0], [1, 1, 0, 2]), ([2, 700000, 699998], [1, 1, 2])):
            want = ref.stream_ops(d, q, w, sizes, ops)
            cuts, pos = [], 0
            for a, op in zip(sizes, ops):
                pos += a
                if op == 1 and pos and (not cuts or cuts[-1] != pos):
                    cuts.append(pos)
            assert _sim_cuts(sim, d, q, w, sizes[0], cuts, [1] * len(cuts), 1) == want, (q, w, sizes)
    d = synth_web(2 * 262144, 9)
    for q, w in ((5, 22), (9, 24)):
        want = ref.stream_ops(d, q, w, [len(d), 0], [0, 2])          # FINISH without input behind full blocks
        assert _sim_cuts(sim, d, q, w, 1 << (18 if q == 9 else 16), [], [], 1, finish_empty=1) == want
        for lgb, dis in ((0, 1), (17, 0), (20, 1), (24, 0)):
            prm = {}
            if lgb:
                prm[3] = lgb
            if dis:
                prm[4] = 1
            want = ref.stream_ops(d, q, w, [len(d)], [2], params=prm)
            assert _sim_cuts(sim, d, q, w, len(d), [], [], 1, lgblock=lgb, disable_ctx=dis) == want, (q, w, lgb, dis)


def _sim_multi(sim, streams, q, w):
    """streams through the device code as ONE batch job (cuts of kind 3); returns the list of compressed streams"""
    sim.sim_compress_multi.restype = C.c_long
    sim.sim_compress_multi.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p,
                                       C.c_size_t, C.c_void_p]
    d = b"".join(streams)
    bounds = np.cumsum([len(x) for x in streams]).astype(np.uint32)
    ends = np.zeros(len(streams) + 1, np.uint64)
    cap = len(d) + len(d) // 2 + 4096 + 64 * len(streams)
    out = C.create_string_buffer(cap)
    st = np.zeros(8, np.uint32)
    r = sim.sim_compress_multi(q, w, d, len(d), bounds.ctypes.data, len(streams), ends.ctypes.data, out, cap, st.ctypes.data)
    assert r >= 0, r
    assert int(ends[len(streams) - 1]) == r
    res, a = [], 0
    for k in range(len(streams)):
        res.append(out.raw[a:int(ends[k])])
        a = int(ends[k])
    return res


def test_sim_batch_of_streams(sim):
    """Many small streams as one device job (br_pipeline.h, cuts of kind 3): every stream must come out exactly as the
    reference compresses it alone -- fresh distance cache / dictionary counters / ring positions at every stream start,
    zero literal contexts in front of it, no match, stitch or merged metablock across a boundary, own window bits."""
    from corpus import synth_binary, synth_text, synth_web
    ora = Oracle()
    rnd = np.random.RandomState(11)
    web = synth_web(700000, 21); txt = synth_text(300000, 22); binr = synth_binary(300000, 23)
    noise = rnd.randint(0, 256, 100000, dtype=np.uint8).tobytes()
    streams = [web[:65536], web[65536:131072], txt[:65536], binr[:65536], noise[:65536], web[131072:131072 + 70000],
               b"a", b"ab", txt[:3], web[:17], bytes(5000), noise[:300], txt[1000:1000 + 65537], web[200000:200000 + 200000],
               binr[100000:100000 + 131072], noise[:40000] + web[:40000], (b"abcdefgh" * 9000)[:66000], web[:65536]]
    for q, w in ((5, 22), (6, 18), (9, 24), (7, 17)):
        got = _sim_multi(sim, streams, q, w)
        for k, x in enumerate(streams):
            assert got[k] == ora.compress(x, q, w), (q, w, k, len(x))
    # streams longer than the ring buffer of a small window (positions wrap relative to the stream start), a bucket with
    # more than 65536 positions of one stream (the reference's uint16 bucket counter wraps), late raw fallbacks
    big = [web[:300000], bytes(150000) + web[:1000] + bytes(100000), web[300000:300000 + 600000], noise[:70000] * 3,
           bytes(rnd.randint(0, 4, 90000, dtype=np.uint8)), web[:100]]
    for q, w in ((5, 17), (8, 18), (6, 22)):
        got = _sim_multi(sim, big, q, w)
        for k, x in enumerate(big):
            assert got[k] == ora.compress(x, q, w), (q, w, k, len(x))
    # several streams that each wrap the counter of the SAME bucket: the count must start at the stream's own first position
    zz = [bytes(200000), bytes(180000) + web[:500] + bytes(90000), b"\x01" * 150000, bytes(70000), web[:100000], bytes(300000)]
    for q, w in ((5, 22), (9, 18)):
        got = _sim_multi(sim, zz, q, w)
        for k, x in enumerate(zz):
            assert got[k] == ora.compress(x, q, w), (q, w, k, len(x))
    # late raw fallbacks (encode.c:604) in many streams of one job: small-alphabet noise passes ShouldCompress and codes
    # larger than its input; every stream's first such metablock is stored raw in the same round (br_assemble_scan)
    fb = []
    for i in range(30):
        n, k = int(rnd.randint(200, 5000)), int(rnd.choice([3, 8, 40, 200, 256]))
        fb.append(bytes(rnd.randint(0, k, n, dtype=np.uint8)) + (web[:int(rnd.randint(1, 300))] if i % 3 == 0 else b""))
    for q, w in ((5, 22), (9, 18)):
        got = _sim_multi(sim, fb, q, w)
        for k, x in enumerate(fb):
            assert got[k] == ora.compress(x, q, w), (q, w, k, len(x))
    # random batches (the last ones with the 2 KiB chunks of a batch that fills the GPU)
    pool = web + txt + binr + noise + bytes(30000)
    for it in range(8):
        if it >= 5:
            os.environ["BR_SIM_BATCH_CHUNK_BITS"] = "11"
        k = int(rnd.randint(2, 40))
        ss = []
        for _ in range(k):
            n = int(rnd.choice([1, 2, 5, 100, 1000, 4096, 20000, 65536, 65536, 70000, 150000]))
            n = max(1, int(n * rnd.uniform(0.5, 1.0)))
            o = int(rnd.randint(0, len(pool) - n))
            ss.append(pool[o:o + n])
        q, w = int(rnd.randint(5, 10)), int(rnd.randint(17, 25))
        try:
            got = _sim_multi(sim, ss, q, w)
        finally:
            os.environ.pop("BR_SIM_BATCH_CHUNK_BITS", None)
        for j, x in enumerate(ss):
            assert got[j] == ora.compress(x, q, w), (it, q, w, j, len(x))


def test_sim_batch_regression_same_launch_flip(sim):
    """fuzz case (35, 22) inside a batch (found by batching the fuzz inputs): a search whose view reaches, through positions
    its own run has just left unstored, into an earlier chunk whose bits flip in the same launch.  The successor count of
    br_commit_bits (taken over the previous snapshot) does not see that far; the bucket is a heavy one and the
    counter-wrap sensitivity of the heavy path (br_lz77.h) re-walks the chunk -- in a batch too, from the stream's first byte."""
    from fuzz_cases import cases
    ora = Oracle()
    d = next(x for i, x, q, w in cases(35, 23) if i == 22)
    other = bytes(np.random.RandomState(1).randint(0, 256, 3000, dtype=np.uint8))
    for bits in ("9", "11"):
        os.environ["BR_SIM_BATCH_CHUNK_BITS"] = bits
        try:
            for ss in ([other, d], [d, other], [d, d]):
                got = _sim_multi(sim, ss, 5, 17)
                assert [got[k] == ora.compress(x, 5, 17) for k, x in enumerate(ss)] == [True] * len(ss), bits
        finally:
            os.environ.pop("BR_SIM_BATCH_CHUNK_BITS", None)


def test_sim_batch_fuzz_sample(sim):
    """The structured fuzz inputs (tests/fuzz_cases.py: periodic, dictionary words, noise, heavy buckets ...) grouped by
    (quality, lgwin) and compressed a dozen at a time as one batch job, with both chunk sizes."""
    import collections
    from fuzz_cases import cases, dict_cases
    ora = Oracle()
    groups = collections.defaultdict(list)
    for src in (cases(4242, 160), dict_cases(4242, 40, TABLES)):
        for i, d, q, w in src:
            if 5 <= q <= 9 and 17 <= w <= 24 and 0 < len(d) < (1 << 20):
                groups[(q, w)].append(d)
    checked = 0
    for (q, w), lst in sorted(groups.items()):
        for a in range(0, len(lst), 12):
            part = lst[a:a + 12]
            if len(part) < 2:
                continue
            os.environ["BR_SIM_BATCH_CHUNK_BITS"] = "11" if (a // 12) % 2 else "9"
            try:
                got = _sim_multi(sim, part, q, w)
            finally:
                os.environ.pop("BR_SIM_BATCH_CHUNK_BITS", None)
            for k, x in enumerate(part):
                assert got[k] == ora.compress(x, q, w), (q, w, a, k, len(x))
                checked += 1
    assert checked > 100


def test_sim_stream_offset(sim):
    """BROTLI_PARAM_STREAM_OFFSET (encode.h:231, the sanctioned way to stitch shards into one stream, SURVEY.md 8e): no
    window bits, poisoned distance cache (encode.c:656), dictionary distances counted from the virtual start
    (backward_references_inc.h:94), and the first two bytes flushed on their own (encode.c:1704) -- against the reference."""
    from brotli_libs import RecordedRef
    from corpus import synth_text, synth_web
    ref = RecordedRef()
    for d in (synth_text(300000, 4), synth_web(500000, 10)):
        for q, w in ((5, 22), (9, 24), (6, 18)):
            for off in (1, 1000, 1 << 20, 1 << 30):
                want = ref.stream_ops(d, q, w, [len(d)], [2], params={9: off})
                got = _sim_cuts(sim, d, q, w, len(d), [2], [1], 1, stream_offset=off, with_header=0)
                assert got == want, (q, w, off, len(got), len(want))


# ---------------------------------------------------------------------------------------------------------------------
# Qualities 2..4 (SURVEY.md 8f rank 1): slot-sorted index + br_find_quick + br_verify_run, flat metablocks at quality 2, 3
from golden_cases import CASES_ORACLE_ONLY

Q234_SMALL = [c for c in CASES_ORACLE_ONLY if c["n"] <= 1_500_000]


@pytest.mark.parametrize("c", Q234_SMALL, ids=lambda c: "%s-%d-q%d-w%d" % (c["kind"], c["n"], c["q"], c["lgwin"]))
def test_sim_q234_matches_oracle(sim, c):
    d = make_case(c)
    want = Oracle().compress(d, c["q"], c["lgwin"])
    cap = len(d) + len(d) // 2 + 4096
    out = C.create_string_buffer(cap)
    st = np.zeros(8, np.uint32)
    r = sim.sim_compress(c["q"], c["lgwin"], d, len(d), out, cap, st.ctypes.data)
    assert r >= 0
    assert out.raw[:r] == want


def test_sim_q234_windows_and_shapes(sim):
    """Small and large windows (lgwin 10..24: window bits of every form, ring smaller than the input block at quality 4),
    the H4 -> H54 switch at 1 MiB, degenerate inputs (long runs: unstored stretches inside one slot, the slot-0 candidate
    of the zeroed table), incompressible input (raw metablocks, sparse-search phases)."""
    from corpus import synth_binary, synth_text, synth_web
    ora = Oracle()
    web = synth_web(1_100_000, 41)
    shapes = [synth_text(180000, 42), synth_binary(250000, 43), web[:(1 << 20) - 1], web[:1 << 20], bytes(300000),
              bytes(range(256)) * 600, np.random.default_rng(44).integers(0, 256, 120000, dtype=np.uint8).tobytes(),
              b"abcdefgh" * 20000 + synth_text(50000, 45) + b"abcdefgh" * 20000]
    for i, d in enumerate(shapes):
        for q in (2, 3, 4):
            for w in ((10, 16, 22) if len(d) < 500000 else (17, 24)):
                assert _fuzz_check(sim, d, q, w), (i, len(d), q, w)


def test_sim_q234_fuzz_sample(sim):
    from fuzz_cases import cases, dict_cases
    for i, d, q, w in cases(20250925, 90):
        if d and len(d) <= 120000:
            q2 = 2 + i % 3
            assert _fuzz_check(sim, d, q2, w), (i, len(d), q2, w)
            assert _fuzz_check(sim, d, q2, 10 + i % 8), (i, len(d), q2, 10 + i % 8)
    for i, d, q, w in dict_cases(20250926, 30, TABLES):     # static-dictionary words: the shallow probe of H2 / H4
        for q2 in (2, 4):
            assert _fuzz_check(sim, d, q2, w), ("dict", i, len(d), q2, w)


def test_sim_q234_flush_cuts(sim):
    """Qualities 2..4 with the input cut by FLUSH operations, against the reference's CompressStream driven with the same
    calls: input blocks of 1 << 14 bytes below quality 4 (quality.h:81), the MAX_NUM_DELAYED_SYMBOLS flush rule
    (encode.c:1152), FINISH without input behind a full block."""
    from brotli_libs import RecordedRef
    from corpus import synth_binary, synth_text
    ref = RecordedRef()
    for d in (synth_text(300000, 3), synth_binary(400000, 5)):
        n = len(d)
        for q, w in ((2, 22), (3, 18), (4, 22), (4, 12)):
            bs = 1 << (14 if q < 4 else 16)
            for sizes, ops in (([100000, 50000, n - 150000], [0, 1, 2]), ([bs, 0, n - bs, 0], [0, 1, 1, 2]), ([100, n - 100, 0], [1, 0, 2])):
                want = ref.stream_ops(d, q, w, sizes, ops)
                pos, cuts, acc, fixed, hint = 0, [], 0, False, 0
                for a, op in zip(sizes, ops):
                    if not fixed and (op != 0 or acc + a >= bs):   # encode.c:1619: the size hint freezes at the first EncodeData
                        hint, fixed = acc + a, True
                    acc += a
                    pos += a
                    if op == 1 and pos > 0 and (not cuts or cuts[-1] != pos):
                        cuts.append(pos)
                if cuts and cuts[-1] == n:
                    got = _sim_cuts(sim, d, q, w, hint, cuts, [1] * len(cuts), 0) + b"\x03"
                else:
                    got = _sim_cuts(sim, d, q, w, hint, cuts, [1] * len(cuts), 1)
                assert got == want, (q, w, sizes, ops)
    d = synth_text(4 * 65536, 9)
    for q, w in ((2, 22), (3, 22), (4, 22)):
        want = ref.stream_ops(d, q, w, [len(d), 0], [0, 2])          # FINISH without input behind full blocks
        assert _sim_cuts(sim, d, q, w, 1 << (14 if q < 4 else 16), [], [], 1, finish_empty=1) == want, (q, w)


def test_sim_q234_batch_of_streams(sim):
    """Qualities 2..4: many small streams as ONE device job (cuts of kind 3).  Slots, window limits and the zeroed-table
    candidate count from every stream's own first byte; every stream must come out as the reference compresses it alone."""
    from corpus import synth_binary, synth_text, synth_web
    ora = Oracle()
    rnd = np.random.RandomState(12)
    web = synth_web(700000, 21); txt = synth_text(300000, 22); binr = synth_binary(300000, 23)
    noise = rnd.randint(0, 256, 100000, dtype=np.uint8).tobytes()
    streams = [web[:65536], web[65536:131072], txt[:65536], binr[:65536], noise[:65536], web[131072:131072 + 70000],
               b"a", b"ab", txt[:3], web[:17], bytes(5000), noise[:300], txt[1000:1000 + 65537], web[200000:200000 + 200000],
               binr[100000:100000 + 131072], noise[:40000] + web[:40000], (b"abcdefgh" * 9000)[:66000], web[:65536]]
    for q, w in ((2, 22), (3, 18), (4, 24), (4, 12), (2, 10), (3, 16)):
        got = _sim_multi(sim, streams, q, w)
        for k, x in enumerate(streams):
            assert got[k] == ora.compress(x, q, w), (q, w, k, len(x))
    zz = [bytes(200000), bytes(180000) + web[:500] + bytes(90000), b"\x01" * 150000, bytes(70000), web[:100000], bytes(300000),
          web[:300000], noise[:70000] * 3, bytes(rnd.randint(0, 4, 90000, dtype=np.uint8))]
    for q, w in ((2, 22), (3, 17), (4, 18)):
        got = _sim_multi(sim, zz, q, w)
        for k, x in enumerate(zz):
            assert got[k] == ora.compress(x, q, w), (q, w, k, len(x))
    fb = []
    for i in range(30):
        n, k = int(rnd.randint(200, 5000)), int(rnd.choice([3, 8, 40, 200, 256]))
        fb.append(bytes(rnd.randint(0, k, n, dtype=np.uint8)) + (web[:int(rnd.randint(1, 300))] if i % 3 == 0 else b""))
    for q, w in ((2, 22), (3, 22), (4, 18)):
        got = _sim_multi(sim, fb, q, w)
        for k, x in enumerate(fb):
            assert got[k] == ora.compress(x, q, w), (q, w, k, len(x))
    pool = web + txt + binr + noise + bytes(30000)
    for it in range(10):
        if it >= 6:
            os.environ["BR_SIM_BATCH_CHUNK_BITS"] = "11"
        k = int(rnd.randint(2, 40))
        ss = []
        for _ in range(k):
            n = int(rnd.choice([1, 2, 5, 100, 1000, 4096, 20000, 65536, 65536, 70000, 150000]))
            n = max(1, int(n * rnd.uniform(0.5, 1.0)))
            o = int(rnd.randint(0, len(pool) - n))
            ss.append(pool[o:o + n])
        q, w = int(rnd.randint(2, 5)), int(rnd.randint(10, 25))
        try:
            got = _sim_multi(sim, ss, q, w)
        finally:
            os.environ.pop("BR_SIM_BATCH_CHUNK_BITS", None)
        for j, x in enumerate(ss):
            assert got[j] == ora.compress(x, q, w), (it, q, w, j, len(x))


def test_sim_q234_batch_fuzz_sample(sim):
    """The structured fuzz inputs a dozen at a time as one batch job at quality 2..4, with both chunk sizes."""
    import collections
    from fuzz_cases import cases, dict_cases
    ora = Oracle()
    groups = collections.defaultdict(list)
    for src in (cases(4243, 150), dict_cases(4243, 40, TABLES)):
        for i, d, q, w in src:
            if 0 < len(d) < 300000:
                groups[(2 + i % 3, 10 + (i * 7) % 15)].append(d)
    checked = 0
    for (q, w), lst in sorted(groups.items()):
        for a in range(0, len(lst), 12):
            part = lst[a:a + 12]
            if len(part) < 2:
                continue
            os.environ["BR_SIM_BATCH_CHUNK_BITS"] = "11" if (a // 12) % 2 else "9"
            try:
                got = _sim_multi(sim, part, q, w)
            finally:
                os.environ.pop("BR_SIM_BATCH_CHUNK_BITS", None)
            for k, x in enumerate(part):
                assert got[k] == ora.compress(x, q, w), (q, w, a, k, len(x))
                checked += 1
    assert checked > 100


def test_sim_q234_index_against_numpy(sim):
    """tests/slot_index.py (the numpy restatement the GPU test checks the three-pass radix sort against) == the sim's index."""
    from corpus import synth_web
    from slot_index import slot_index
    sim.sim_debug_sort.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_uint32, C.c_void_p, C.c_void_p]
    for q, n in ((2, 300000), (3, 300000), (4, 300000), (4, 1 << 20), (4, 5000), (2, 9), (3, 7)):
        d = synth_web(n, 17)
        want_S, want_seg, bits = slot_index(d, q)
        S = np.zeros(n, np.uint32); seg = np.zeros((1 << bits) + 2, np.uint32)
        assert sim.sim_debug_sort(q, 22, d, n, S.ctypes.data, seg.ctypes.data)
        assert np.array_equal(S, want_S), (q, n)
        assert np.array_equal(seg, want_seg), (q, n)


def test_sim_flush_just_behind_a_block_boundary(sim):
    """A FLUSH one or two bytes (up to HashTypeLength - 2) behind a block boundary leaves an input block too short to stitch
    (hash_longest_match_quickly_inc.h:119 / hash_longest_match64_inc.h:127: num_bytes >= HashTypeLength - 1); the block behind
    it stitches instead, and its three positions reach back across the short block into the block in front.  Their owner must
    still commit them (br_commit_bits; found by a randomized FLUSH campaign: q3, lgwin 12, flush at 14 * 16384 + 2)."""
    from brotli_libs import RecordedRef
    from corpus import synth_text
    ref = RecordedRef()
    d = synth_text(200000, 77)
    n = len(d)
    for q, w in ((3, 12), (2, 22), (4, 16), (5, 22), (7, 17)):
        bs = 1 << (14 if q < 4 else 16)
        for extra in (1, 2, 3, 5, 6):
            c = 2 * bs + extra
            want = ref.stream_ops(d, q, w, [c, n - c], [1, 2])
            assert _sim_cuts(sim, d, q, w, c, [c], [1], 1) == want, (q, w, extra)
        c1, c2 = bs + 1, bs + 2                                    # two short blocks in a row
        want = ref.stream_ops(d, q, w, [c1, 1, n - c2], [1, 1, 2])
        assert _sim_cuts(sim, d, q, w, c1, [c1, c2], [1, 1], 1) == want, (q, w)
