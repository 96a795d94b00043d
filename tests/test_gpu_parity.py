"""GPU suite (-m gpu): the CUDA path, called through the C ABI, against the golden vectors of the
compiled reference, the oracle, and the reference's recorded outputs (brotli_libs.RecordedRef).  Bit-exact."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

from brotli_libs import Oracle, RecordedRef
from golden_cases import make_case

pytestmark = pytest.mark.gpu
GOLDEN = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden.json")))


@pytest.fixture(scope="module")
def b200():
    import brotli_b200
    assert brotli_b200.available(), "no CUDA device"
    return brotli_b200


@pytest.mark.parametrize("g", GOLDEN, ids=lambda g: "%s-%d-q%d-w%d" % (g["kind"], g["n"], g["q"], g["lgwin"]))
def test_golden(b200, g):
    d = make_case(g)
    assert hashlib.sha256(d).hexdigest() == g["in_sha256"]
    out = b200.compress_oneshot(d, g["q"], g["lgwin"])
    assert len(out) == g["out_len"]
    assert hashlib.sha256(out).hexdigest() == g["out_sha256"]


FIXDIR = os.path.join(os.path.dirname(__file__), "golden", "fixtures")
FIXTURES = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "fixtures.json")))


@pytest.mark.parametrize("g", FIXTURES, ids=lambda g: "%s-q%d-w%d" % (g["label"], g["q"], g["lgwin"]))
def test_reference_fixtures(b200, g):
    """The CUDA path on the reference's own tests/testdata files (real text, binary AST, map tiles, repeats, noise,
    a one-byte file ...), against digests of the compiled reference.  alice29.txt[:65536] at quality 5 / lgwin 22 is
    BASELINE.json config C1: 24 091 bytes."""
    d = open(os.path.join(FIXDIR, g["file"]), "rb").read()[:g["n"]]
    assert hashlib.sha256(d).hexdigest() == g["in_sha256"]
    out = b200.compress_oneshot(d, g["q"], g["lgwin"])
    assert len(out) == g["out_len"]
    assert hashlib.sha256(out).hexdigest() == g["out_sha256"]
    if g["label"] == "alice29.txt[:65536]" and g["q"] == 5:
        assert len(out) == 24091


def test_against_oracle_all_qualities(b200):
    ora = Oracle()
    from corpus import synth_text, synth_web
    d1, d2 = synth_text(700000, 31), synth_web(1300000, 32)
    for q in (5, 6, 7, 8, 9):
        for w in (17, 19, 22, 24):
            for d in (d1, d2):
                assert b200.compress_oneshot(d, q, w) == ora.compress(d, q, w), (q, w, len(d))


def test_edge_sizes(b200):
    ora = Oracle()
    from corpus import synth_text
    base = synth_text(200000, 33)
    for n in (1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 63, 64, 65, 511, 512, 4095, 65535, 65536, 65537, 131072, 131073):
        d = base[:n]
        assert b200.compress_oneshot(d, 5, 22) == ora.compress(d, 5, 22), n
        assert b200.compress_oneshot(d, 9, 24) == ora.compress(d, 9, 24), n
    assert b200.compress_oneshot(b"", 5, 22) == b"\x06"


def test_streaming_api_equals_oneshot(b200):
    from corpus import synth_text
    d = synth_text(1500000, 34)
    want = Oracle().compress(d, 5, 22)
    c = b200.Compressor(quality=5, lgwin=22)
    out = b""
    # first call carries everything: the size hint freezes at the full length like the one-shot call
    out += c.process(d)
    out += c.finish()
    assert out == want
    assert b200.compress(d, quality=5, lgwin=22) == want
    # empty stream through the streaming API
    c2 = b200.Compressor(quality=5, lgwin=22)
    assert c2.finish() == bytes([0x3B])   # window bits 1011 + ISLAST + ISEMPTY (encode.c:1006)


def _drive(b200, d, q, w, sizes, ops):
    """The same (size, op) call sequence through this library's streaming API."""
    c = b200.Compressor(quality=q, lgwin=w)
    out, pos = b"", 0
    for a, op in zip(sizes, ops):
        out += c._stream(d[pos:pos + a], op)
        pos += a
    return out


def test_streaming_flush_and_metadata(b200):
    """FLUSH and EMIT_METADATA at quality 5..9 (encode.c:1356, :1549): byte-identical to the reference's CompressStream for
    the same call sequence -- flushes inside and at block boundaries, a flush / metadata before any input, metadata between
    data, repeated operations at one position, FINISH without input behind a full block, and everything flushed bytewise."""
    from corpus import synth_binary, synth_text
    ref = RecordedRef()
    for d in (synth_text(700000, 61), synth_binary(900000, 62)):
        n = len(d)
        for q, w in ((5, 22), (9, 24), (6, 18)):
            bs = 1 << (18 if q >= 9 else 16)
            seqs = [
                ([100000, 50000, 250000, n - 400000], [0, 1, 1, 2]),
                ([0, 300000, 0, n - 300000, 0], [1, 1, 1, 1, 2]),
                ([bs, 0, n - bs], [0, 1, 2]),
                ([2 * bs, 0], [0, 2]),
                ([7, 200000, 5, n - 200012, 0], [3, 0, 3, 1, 2]),          # metadata first (payload = the input bytes), between data
                ([0, 100, 0, 0, 11, n - 111], [3, 1, 3, 1, 3, 2]),        # empty metadata, repeated operations at one position
            ]
            for sizes, ops in seqs:
                if sum(a for a, op in zip(sizes, ops) if op != 3) > n:
                    continue
                # metadata payloads are taken from the same buffer; they are not stream input
                want = ref.stream_ops(d, q, w, sizes, ops)
                got = _drive(b200, d, q, w, sizes, ops)
                assert got == want, (q, w, sizes, ops, len(got), len(want))
                # the flushed prefixes really decode: cut the stream behind its last flush and finish it by hand
    # FLUSH makes the data so far decodable (encode.h:105): check on one sequence with the reference decoder
    d = synth_text(300000, 63)
    c = b200.Compressor(quality=5, lgwin=22)
    part = c.process(d[:200000]) + c.flush()
    assert ref.decompress(part + b"\x03", 200000) == d[:200000]      # ISLAST + ISEMPTY appended on the byte boundary
    rest = c.process(d[200000:]) + c.finish()
    assert ref.decompress(part + rest, len(d)) == d


def test_lgblock_and_context_modeling_parameters(b200):
    """BROTLI_PARAM_LGBLOCK (encode.h:184, quality.h:76) and BROTLI_PARAM_DISABLE_LITERAL_CONTEXT_MODELING (encode.h:191,
    encode.c:561) through the streaming API, against the reference with the same parameters."""
    from corpus import synth_web
    ref = RecordedRef()
    L = b200.lib()
    d = synth_web(1500000, 65)
    for q, w in ((5, 22), (9, 24)):
        for lgb, dis in ((0, 1), (17, 0), (20, 1), (24, 0)):
            prm = {}
            if lgb:
                prm[3] = lgb
            if dis:
                prm[4] = 1
            want = ref.stream_ops(d, q, w, [700000, len(d) - 700000], [1, 2], params=prm)
            c = b200.Compressor(quality=q, lgwin=w, lgblock=lgb)
            if dis:
                assert L.BrotliEncoderSetParameter(c._s, 4, 1)
            got = c._stream(d[:700000], 1) + c._stream(d[700000:], 2)
            assert got == want, (q, w, lgb, dis)


def test_stream_offset_stitches_shards(b200):
    """SURVEY.md 8e: one valid stream out of independently compressed shards -- every shard but the first is compressed with
    BROTLI_PARAM_STREAM_OFFSET = its start (encode.h:231), every shard but the last ends with FLUSH instead of FINISH.
    Each shard equals the reference run with the same parameters and calls; the concatenation decodes to the input."""
    from corpus import synth_web
    ref = RecordedRef()
    L = b200.lib()
    d = synth_web(1800000, 68)
    cuts = [0, 500000, 1300001, len(d)]
    for q, w in ((5, 22), (9, 24)):
        whole = b""
        for i in range(3):
            part = d[cuts[i]:cuts[i + 1]]
            last = i == 2
            prm = {9: cuts[i]} if i else {}
            want = ref.stream_ops(part, q, w, [len(part)], [2 if last else 1], params=prm)
            c = b200.Compressor(quality=q, lgwin=w)
            if i:
                # (the Compressor has not been used yet: parameters can still be set)
                assert L.BrotliEncoderSetParameter(c._s, 9, cuts[i])
            got = c._stream(part, 2 if last else 1)
            assert got == want, (q, w, i, len(got), len(want))
            whole += got
        assert ref.decompress(whole, len(d)) == d


def test_custom_allocator(b200):
    """encode.h:295: an instance created with an allocator pair takes its memory (state and buffers) from it."""
    L = b200.lib()
    ALLOC = C.CFUNCTYPE(C.c_void_p, C.c_void_p, C.c_size_t)
    FREE = C.CFUNCTYPE(None, C.c_void_p, C.c_void_p)
    libc = C.CDLL(None)
    libc.malloc.restype = C.c_void_p; libc.malloc.argtypes = [C.c_size_t]; libc.free.argtypes = [C.c_void_p]
    stat = {"allocs": 0, "frees": 0, "bytes": 0}

    def a(opaque, n):
        stat["allocs"] += 1; stat["bytes"] += n
        return libc.malloc(n)

    def f(opaque, p):
        if p:
            stat["frees"] += 1
            libc.free(p)
    af, ff = ALLOC(a), FREE(f)
    L.BrotliEncoderCreateInstance.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    assert not L.BrotliEncoderCreateInstance(C.cast(af, C.c_void_p), None, None)     # both or neither
    st = L.BrotliEncoderCreateInstance(C.cast(af, C.c_void_p), C.cast(ff, C.c_void_p), None)
    assert st
    from corpus import synth_text
    d = synth_text(400000, 64)
    L.BrotliEncoderSetParameter(st, 1, 5); L.BrotliEncoderSetParameter(st, 2, 22)
    buf = C.create_string_buffer(d, len(d))
    avail_in = C.c_size_t(len(d)); next_in = C.c_void_p(C.addressof(buf))
    avail_out = C.c_size_t(0); next_out = C.c_void_p(None)
    assert L.BrotliEncoderCompressStream(st, 2, C.byref(avail_in), C.byref(next_in), C.byref(avail_out), C.byref(next_out), None)
    out = b""
    while L.BrotliEncoderHasMoreOutput(st):
        sz = C.c_size_t(0)
        p = L.BrotliEncoderTakeOutput(st, C.byref(sz))
        out += C.string_at(p, sz.value)
    L.BrotliEncoderDestroyInstance(st)
    assert out == Oracle().compress(d, 5, 22)
    assert stat["allocs"] >= 3 and stat["bytes"] >= len(d) and stat["allocs"] == stat["frees"]


def test_device_and_batch_api(b200):
    import torch
    from corpus import synth_text, synth_web
    ora = Oracle()
    L = b200.lib()
    d = synth_text(2000000, 35)
    want = ora.compress(d, 5, 22)
    t = torch.frombuffer(bytearray(d), dtype=torch.uint8).cuda()
    out = torch.empty(len(d) + 4096, dtype=torch.uint8, device="cuda")
    sz = C.c_size_t(out.numel())
    assert L.BrotliB200CompressDevice(5, 22, len(d), t.data_ptr(), C.byref(sz), out.data_ptr())
    assert bytes(out[:sz.value].cpu().numpy().tobytes()) == want
    # batch of independent streams over 4 host workers
    ins = [synth_web(100000 + 7777 * i, 40 + i) for i in range(12)]
    bufs = [C.create_string_buffer(len(x) + 4096) for x in ins]
    inp = (C.c_void_p * 12)(*[C.cast(C.c_char_p(x), C.c_void_p) for x in ins])
    outp = (C.c_void_p * 12)(*[C.cast(b, C.c_void_p) for b in bufs])
    isz = (C.c_size_t * 12)(*[len(x) for x in ins])
    osz = (C.c_size_t * 12)(*[len(x) + 4096 for x in ins])
    assert L.BrotliB200CompressBatch(5, 22, 12, inp, isz, outp, osz, 4) == 12
    for i in range(12):
        assert bufs[i].raw[:osz[i]] == ora.compress(ins[i], 5, 22), i


def test_batch_of_small_streams(b200):
    """BrotliB200CompressBatch at quality 5..9: streams below 1 MiB run as ONE device job per group (streams laid end to
    end, cuts of kind 3 in br_pipeline.h); every stream must equal what BrotliEncoderCompress gives for it alone -- sizes
    1 byte .. 900 KB, empty streams, streams above 1 MiB in the same call, incompressible ones (raw fallback, raw-stream
    rule), long zero runs (bucket counter wrap), windows smaller than the stream."""
    from corpus import synth_binary, synth_text, synth_web
    ora = Oracle()
    rnd = np.random.RandomState(17)
    web = synth_web(3_000_000, 81); txt = synth_text(1_000_000, 82); binr = synth_binary(1_000_000, 83)
    noise = rnd.randint(0, 256, 200000, dtype=np.uint8).tobytes()
    pool = web + txt + binr + noise + bytes(200000)
    streams = [web[:65536], b"", b"a", web[:3], noise[:300], noise[:65536], bytes(150000) + web[:1000] + bytes(100000), web[:900000],
               web[100000:100000 + 1_200_000], txt[:65537], binr[:262144], (b"abcdefgh" * 9000)[:66000], noise[:70000] * 3]
    for _ in range(120):
        n = int(rnd.choice([1, 2, 5, 100, 1000, 4096, 20000, 65536, 65536, 65536, 70000, 150000, 400000]))
        n = max(1, int(n * rnd.uniform(0.5, 1.0)))
        o = int(rnd.randint(0, len(pool) - n))
        streams.append(pool[o:o + n])
    for q, w in ((5, 22), (9, 24), (6, 17), (7, 18)):
        got = b200.compress_batch(streams, q, w, threads=4)
        for k, x in enumerate(streams):
            assert got[k] == ora.compress(x, q, w), (q, w, k, len(x))
    # 20 000 tiny streams (1 .. 2 000 bytes): several groups of at most 8 192 streams (br_api.cc kBatchGroupStreams)
    tiny = []
    for _ in range(20000):
        n = int(rnd.choice([1, 2, 3, 7, 30, 200, 700, 2000]))
        o = int(rnd.randint(0, len(pool) - n))
        tiny.append(pool[o:o + n])
    got = b200.compress_batch(tiny, 5, 22, threads=4)
    for k, x in enumerate(tiny):
        assert got[k] == ora.compress(x, 5, 22), (k, len(x))
    # a batch that fills the GPU takes the 2 KiB chunks (br_params.h br_batch_chunk_bits): 400 x 64 KiB
    big = [pool[o:o + 65536] for o in [(i * 104729) % (len(pool) - 65536) for i in range(400)]]
    got = b200.compress_batch(big, 5, 22, threads=4)
    for k, x in enumerate(big):
        assert got[k] == ora.compress(x, 5, 22), k


def test_full_size_properties(b200):
    """BASELINE.json's full size (100 MB, q5, lgwin 22): equality with the reference's output,
    and the size-independent property decode(encode(x)) == x via the reference decoder (both recorded)."""
    from corpus import synth_text
    ref = RecordedRef()
    d = synth_text(100_000_000)
    out = b200.compress_oneshot(d, 5, 22)
    assert ref.decompress(out, len(d)) == d
    assert out == ref.compress(d, 5, 22)


def test_q9_ring_wrap_and_nonsettling_inputs(b200):
    """Quality 9 / lgwin 24 beyond the 32 MiB ring buffer of the reference (BASELINE config C4's path: H6, 256-entry
    rings, 256 KiB input blocks), on the Silesia-shaped binary mix, and inputs whose parse never settles by itself --
    uniform noise (the sparse search's position phase runs through the whole input) and int32 random walks.  The
    encoder must never fail (encode.c:1340-1353) and must equal the reference's output (recorded)."""
    import numpy as np
    from corpus import synth_binary
    ref = RecordedRef()
    cases = [("binary mix 48 MiB", synth_binary(48 << 20, 91), 9, 24),
             ("uniform noise 24 MiB", np.random.RandomState(92).randint(0, 256, 24 << 20, dtype=np.uint8).tobytes(), 9, 24),
             ("uniform noise 16 MiB q5", np.random.RandomState(93).randint(0, 256, 16 << 20, dtype=np.uint8).tobytes(), 5, 22),
             ("random walk 64 MiB", np.cumsum(np.random.RandomState(94).normal(0, 50, (64 << 20) // 4).astype(np.int64)).astype(np.int32).tobytes(), 9, 24)]
    for name, d, q, w in cases:
        out = b200.compress_oneshot(d, q, w)
        assert out == ref.compress(d, q, w), name


def test_config3_slice_and_config5_streams(b200):
    """BASELINE config C3 (web mix, quality 5, lgwin 22) on a 256 MiB slice, and config C5 on 1000 of its 64 KiB streams
    (quality 1, one device batch), each against the reference's recorded outputs."""
    from corpus import synth_web
    ref = RecordedRef()
    web = synth_web(256 << 20)
    out = b200.compress_oneshot(web, 5, 22)
    assert out == ref.compress(web, 5, 22)
    streams = [web[o:o + 65536] for o in [(i * 104729) % (len(web) - 65536) for i in range(1000)]]
    got = b200.compress_batch(streams, 1, 22)
    for i, s in enumerate(streams):
        assert got[i] == ref.compress(s, 1, 22), i


def _check_cli(b200, data, q, w, from_file):
    """The reference's CLI (c/tools/brotli.c, unmodified) on `data` with `-q q -w w`: what it writes when linked against this
    library must equal what it writes when linked against the reference encoder (recorded).  The CLI linked against this
    library (oracle/_ref/brotli_cli_b200) runs where build() could compile it from the reference; the CLI's own call
    loop (brotli_libs.cli_compress_stream: 512 KiB reads, a 512 KiB output buffer drained when full, the size hint of an
    input file) runs over this library everywhere."""
    from brotli_libs import B200_CLI, cli_compress_stream, run_cli
    args = ["-q", str(q), "-w", str(w)]
    want = RecordedRef().cli(args, data, from_file)
    assert len(want) > 0
    got = cli_compress_stream(b200.lib(), data, q, w, 1 << 19, size_hint=len(data) if from_file else 0)
    assert got == want, ("CLI call loop", len(data), q, w, from_file)
    if os.path.exists(B200_CLI):
        assert run_cli(B200_CLI, args, data, from_file) == want, ("brotli_cli_b200", len(data), q, w, from_file)


def test_cli_dropin(b200):
    """The reference's own CLI (c/tools/brotli.c, unmodified) linked against this library instead of libbrotlienc
    produces the same file as the CLI linked against the reference encoder (_check_cli)."""
    from corpus import synth_text
    _check_cli(b200, synth_text(3_000_000, 77), 5, 22, True)


def test_cli_dropin_stdin(b200):
    """The same CLI reading a PIPE: no size hint (c/tools/brotli.c:1448-1452), 512 KiB PROCESS calls, an input that is an
    exact multiple of the read size (FINISH arrives without input behind a full block), quality 5 and 9."""
    from corpus import synth_web
    for n, q, w in ((3 * 524288, 5, 22), (2_500_001, 9, 24), (700_000, 6, 18)):
        _check_cli(b200, synth_web(n, 78), q, w, False)


def test_one_shot_wrapper_rules(b200):
    """encode.c:1296-1353 / quality.h:60: quality 1 with lgwin above 24 is sanitised to 24 (no large window at quality <= 2);
    an output buffer that is too small fails; an incompressible input still fits BrotliEncoderMaxCompressedSize."""
    import numpy as np
    from corpus import synth_text
    ref = RecordedRef()
    L = b200.lib()
    d = synth_text(200000, 66)
    assert b200.compress_oneshot(d, 1, 27) == ref.compress(d, 1, 27) == ref.compress(d, 1, 24)
    noise = np.random.RandomState(67).randint(0, 256, 300000, dtype=np.uint8).tobytes()
    for q, w in ((1, 22), (5, 22), (9, 24)):
        got = b200.compress_oneshot(noise, q, w)
        assert got == ref.compress(noise, q, w) and len(got) <= L.BrotliEncoderMaxCompressedSize(len(noise))
    out = C.create_string_buffer(1000)
    n = C.c_size_t(1000)
    assert L.BrotliEncoderCompress(5, 22, 0, len(d), d, C.byref(n), out) == 0 and n.value == 0     # too small: FALSE, size 0


def test_q1_oneshot_against_oracle(b200):
    """Quality 1 through BrotliEncoderCompress: every hash-table size / min_match, block and fragment
    boundaries, raw meta-blocks, the raw-stream rule."""
    ora = Oracle()
    from corpus import synth_binary, synth_text, synth_web
    base = synth_web(3_000_000, 51)
    for n in (0, 1, 15, 16, 17, 255, 256, 257, 1000, 5000, 40000, 65535, 65536, 65537, 131072, 131073, 300000, 1 << 20, 3_000_000):
        for w in (10, 16, 18, 22, 24):
            assert b200.compress_oneshot(base[:n], 1, w) == ora.compress(base[:n], 1, w), (n, w)
    rnd = np.random.RandomState(5).randint(0, 256, 500000, dtype=np.uint8).tobytes()
    for d in (synth_text(1_400_000, 52), synth_binary(1_400_000, 53), bytes(300000), rnd, rnd[:70000] + bytes(70000) + rnd[:70000]):
        for w in (12, 17, 22):
            assert b200.compress_oneshot(d, 1, w) == ora.compress(d, 1, w), (len(d), w)


def test_q1_batch_c5_shape(b200):
    """BASELINE config C5 in small: many independent 64 KiB streams, quality 1, one device batch; plus
    ragged and empty members."""
    ora = Oracle()
    from corpus import synth_web
    src = synth_web(6_000_000, 54)
    offs = [(i * 104729) % (len(src) - 65536) for i in range(300)]
    streams = [src[o:o + 65536] for o in offs]
    streams += [b"", b"x", src[:15], src[:16], src[:17], src[:100000], src[:300001], bytes(5000),
                np.random.RandomState(6).randint(0, 256, 20000, dtype=np.uint8).tobytes()]
    got = b200.compress_batch(streams, 1, 22)
    assert len(got) == len(streams)
    for i, (g, d) in enumerate(zip(got, streams)):
        assert g == ora.compress(d, 1, 22), i
    st = b200.last_stats_q1()
    assert st["streams"] == len(streams) and st["launches"] > 0


def test_q1_streaming_call_pattern(b200):
    """Quality 1 cuts fragments per CompressStream call: Compressor.process() chunks must give the
    bytes the reference gives for the same calls."""
    from corpus import synth_web
    ora = Oracle()
    d = synth_web(1_700_000, 55)
    for sizes in ([1_700_000], [524288, 524288, 524288, 127136], [1, 15, 16, 17, 1_699_951], [600000, 0, 1_100_000]):
        c = b200.Compressor(quality=1, lgwin=22)
        out, o = b"", 0
        for a in sizes:
            out += c.process(d[o:o + a]); o += a
        out += c.finish()
        calls = [a for a in sizes if a] + [0]
        assert out == ora.compress_q1_stream(d, 22, calls), sizes
    ref = RecordedRef()
    c = b200.Compressor(quality=1, lgwin=18)
    out = b""
    for o in range(0, len(d), 1 << 19):
        out += c.process(d[o:o + (1 << 19)])
    out += c.finish()
    assert out == ref.compress_stream(d, 1, 18, 1 << 19)
    assert ref.decompress(out, len(d)) == d


def test_q1_cli_dropin(b200):
    from corpus import synth_web
    for n in (3_000_000, 1 << 20):       # the second one ends exactly on a 512 KiB read: empty FINISH call
        _check_cli(b200, synth_web(n, 78), 1, 22, True)


def test_q1_flush(b200):
    """Compressor.flush() at quality 1 (go/cbrotli Writer.Flush, encoder_jni FLUSH): bytes delivered by each
    flush are decodable so far and the whole stream equals the reference's for the same op sequence."""
    from corpus import synth_web
    ora = Oracle()
    d = synth_web(900000, 61)
    cases = [([0, 900000], [1, 2]), ([100000, 0, 800000, 0], [1, 1, 1, 2]), ([1, 2, 3, 899994], [1, 1, 0, 2]),
             ([300000, 300000, 300000], [0, 1, 2]), ([450000, 450000, 0], [1, 1, 2])]
    for sizes, ops in cases:
        for w in (16, 22):
            c = b200.Compressor(quality=1, lgwin=w)
            out, o = b"", 0
            for a, op in zip(sizes, ops):
                piece = d[o:o + a]; o += a
                if op == 0:
                    out += c.process(piece)
                elif op == 1:
                    out += c._stream(piece, c._FLUSH)
                else:
                    out += c._stream(piece, c._FINISH)
            assert out == ora.compress_q1_stream(d, w, sizes, ops), (sizes, ops, w)
            assert out == RecordedRef().stream_ops(d, 1, w, sizes, ops)


def test_q1_stream_beyond_one_device_segment(b200):
    """Quality 1 has no stream-size limit: input above one device segment (128 MiB) runs as several, a segment that
    neither flushes nor finishes ends mid-byte and the next starts behind its pending bits (br_api.cc q1_run).
    300 MB in one call (split at multiples of the fragment size) and in 24 MiB + 1 calls (a segment every 64 MiB)."""
    from corpus import synth_web
    rng = np.random.default_rng(77)
    base = np.frombuffer(synth_web(8 << 20, 71), np.uint8)
    d = np.tile(base, 37)[:300_000_000].copy()
    idx = rng.integers(0, d.size, d.size // 50)
    d[idx] = rng.integers(0, 256, idx.size, dtype=np.uint8)
    d[(1 << 27) - 3_000_000:(1 << 27) + 3_000_000] = rng.integers(0, 256, 6_000_000, dtype=np.uint8)   # raw fragments across a cut
    d = d.tobytes()
    ref = RecordedRef()
    for w in (22, 18):
        assert b200.compress_oneshot(d, 1, w) == ref.compress(d, 1, w), w
    step = (24 << 20) + 1
    sizes = [min(step, len(d) - o) for o in range(0, len(d), step)] + [0]
    ops = [0] * (len(sizes) - 1) + [2]
    c = b200.Compressor(quality=1, lgwin=22)
    out, o = [], 0
    for a, op in zip(sizes, ops):
        piece = d[o:o + a]; o += a
        out.append(c.process(piece) if op == 0 else c._stream(piece, c._FINISH))
    assert b"".join(out) == ref.stream_ops(d, 1, 22, sizes, ops)


def test_fuzz_gpu(b200):
    """Structured random inputs (tests/fuzz_cases.py) through the C ABI on the GPU, plus the regression inputs."""
    from fuzz_cases import REGRESSIONS, cases
    ora = Oracle()
    todo = []
    by_seed = {}
    for seed, idx in REGRESSIONS:
        by_seed.setdefault(seed, set()).add(idx)
    for seed, idxs in by_seed.items():
        todo += [(seed, i, d, q, w) for i, d, q, w in cases(seed, max(idxs) + 1) if i in idxs]
    todo += [(31337, i, d, q, w) for i, d, q, w in cases(31337, 250)]
    for seed, i, d, q, w in todo:
        assert b200.compress_oneshot(d, q, w) == ora.compress(d, q, w), (seed, i, len(d), q, w)
