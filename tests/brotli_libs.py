"""ctypes loaders for the checker libraries (oracle/ and oracle/_ref) and the product
C-ABI (brotli_b200/libbrotlienc_b200.so), and RecordedRef, the reference's recorded
outputs the suite compares against.  Test infrastructure only."""
import atexit
import ctypes as C
import hashlib
import json
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libbrotli_ref.so")
REF_CLI = os.path.join(ROOT, "oracle", "_ref", "brotli_cli_ref")
B200_CLI = os.path.join(ROOT, "oracle", "_ref", "brotli_cli_b200")    # the same CLI linked against this library
PROBE_SO = os.path.join(ROOT, "oracle", "_ref", "libbrotli_probe.so")
ORACLE_SO = os.path.join(ROOT, "oracle", "liboracle.so")
TABLES = os.path.join(ROOT, "brotli_b200", "data", "brotli_tables.bin")
PRODUCT_SO = os.path.join(ROOT, "brotli_b200", "libbrotlienc_b200.so")
REFERENCE_OUTPUTS = os.path.join(ROOT, "tests", "golden", "reference_outputs.json")

_u8p = C.POINTER(C.c_uint8)


def _buf(b):
    return (C.c_uint8 * max(1, len(b))).from_buffer_copy(b if len(b) else b"\0")


def zeroed_malloc():
    """The reference reads ring-buffer bytes it never wrote in some call sequences (c/enc/ringbuffer.h:104-116: the first write
    of less than a block skips the tail copy, and the buffer is grown by a plain malloc, :70-78; a later block that runs across
    the ring's end then compares against tail bytes nobody filled), so its output depends on what malloc hands out: identical
    in a fresh process (zero pages), different on a dirty heap (found by tools/sim_campaign.py: quality 4, lgwin 10, three
    FLUSHes; MALLOC_PERTURB_ flips it).  This makes malloc hand out zeroed memory in the calling process -- what a fresh
    process gets and what the oracle models (stale_byte) -- so that comparisons do not flake.  Called by tests/conftest.py and
    the campaign tools only: bench.py must time the reference with the allocator as it is."""
    try:
        C.CDLL(None).mallopt(-6, 255)      # M_PERTURB: allocations are filled with ~255 = 0
    except Exception:
        pass


class Ref:
    """The unmodified reference, compiled from its sources into oracle/_ref by oracle/Makefile."""

    def __init__(self, path=REF_SO):
        self.lib = C.CDLL(path, mode=os.RTLD_LOCAL)
        L = self.lib
        L.BrotliEncoderCompress.argtypes = [C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_void_p,
                                            C.POINTER(C.c_size_t), C.c_void_p]
        L.BrotliEncoderCompress.restype = C.c_int
        L.BrotliEncoderMaxCompressedSize.argtypes = [C.c_size_t]
        L.BrotliEncoderMaxCompressedSize.restype = C.c_size_t
        L.BrotliDecoderDecompress.argtypes = [C.c_size_t, C.c_void_p, C.POINTER(C.c_size_t), C.c_void_p]
        L.BrotliDecoderDecompress.restype = C.c_int

    def compress(self, data, quality, lgwin, mode=0):
        n = len(data)
        cap = self.lib.BrotliEncoderMaxCompressedSize(n) + 16
        out = C.create_string_buffer(cap)
        out_n = C.c_size_t(cap)
        ok = self.lib.BrotliEncoderCompress(quality, lgwin, mode, n, data, C.byref(out_n), out)
        assert ok == 1
        return out.raw[:out_n.value]

    def decompress(self, comp, max_out):
        out = C.create_string_buffer(max(1, max_out))
        out_n = C.c_size_t(max_out)
        ok = self.lib.BrotliDecoderDecompress(len(comp), comp, C.byref(out_n), out)
        assert ok == 1, "decoder rejected the stream"
        return out.raw[:out_n.value]


class Oracle:
    """Our CPU restatement (oracle/brotli_oracle.c)."""

    def __init__(self, path=ORACLE_SO):
        self.lib = C.CDLL(path, mode=os.RTLD_LOCAL)
        L = self.lib
        L.oracle_init.argtypes = [C.c_void_p, C.c_size_t]
        L.oracle_init.restype = C.c_int
        L.oracle_brotli_compress.argtypes = [C.c_int, C.c_int, C.c_size_t, C.c_void_p,
                                             C.POINTER(C.c_size_t), C.c_void_p]
        L.oracle_brotli_compress.restype = C.c_int
        L.oracle_fast_log2.argtypes = [C.c_size_t]
        L.oracle_fast_log2.restype = C.c_double
        blob = open(TABLES, "rb").read()
        assert L.oracle_init(blob, len(blob)) == 1

    def compress_q1_stream(self, data, lgwin, calls=None, ops=None):
        """The quality-1 stream for a sequence of CompressStream calls (sizes, and optionally their
        operations: 0 PROCESS, 1 FLUSH, 2 FINISH); None = one FINISH call."""
        L = self.lib
        L.oracle_brotli_compress_q1_ops.argtypes = [C.c_int, C.c_size_t, C.c_char_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                                    C.POINTER(C.c_size_t), C.c_void_p]
        cap = 2 * len(data) + 100000
        out = C.create_string_buffer(cap)
        n = C.c_size_t(cap)
        arr = (C.c_size_t * len(calls))(*calls) if calls is not None else None
        oarr = (C.c_int * len(ops))(*ops) if ops is not None else None
        assert L.oracle_brotli_compress_q1_ops(lgwin, len(data), data, len(calls) if calls is not None else 0, arr, oarr,
                                               C.byref(n), out) == 1
        return out.raw[:n.value]

    def compress(self, data, quality, lgwin):
        n = len(data)
        cap = n + (n >> 1) + 4096
        out = C.create_string_buffer(cap)
        out_n = C.c_size_t(cap)
        ok = self.lib.oracle_brotli_compress(quality, lgwin, n, data, C.byref(out_n), out)
        assert ok == 1
        return out.raw[:out_n.value]


def cli_compress_stream(L, data, quality, lgwin, chunk, out_buf=1 << 19, size_hint=0):
    """Drives the streaming API of library L (the reference's or this project's) the way c/tools/brotli.c:1357 does:
    PROCESS calls of `chunk` bytes, FINISH once the input is exhausted (an extra empty call when the size is a multiple
    of `chunk`, like feof() after a full read), a caller output buffer of `out_buf` bytes drained whenever it is full,
    until BrotliEncoderIsFinished; `size_hint` as the CLI sets it for an input file (c/tools/brotli.c:1448)."""
    L.BrotliEncoderCreateInstance.restype = C.c_void_p
    L.BrotliEncoderCreateInstance.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.BrotliEncoderSetParameter.argtypes = [C.c_void_p, C.c_int, C.c_uint32]
    L.BrotliEncoderDestroyInstance.argtypes = [C.c_void_p]
    L.BrotliEncoderIsFinished.argtypes = [C.c_void_p]
    L.BrotliEncoderCompressStream.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_size_t), C.POINTER(C.c_void_p),
                                              C.POINTER(C.c_size_t), C.POINTER(C.c_void_p), C.c_void_p]
    s = L.BrotliEncoderCreateInstance(None, None, None)
    L.BrotliEncoderSetParameter(s, 1, quality)
    L.BrotliEncoderSetParameter(s, 2, lgwin)
    if size_hint:
        L.BrotliEncoderSetParameter(s, 5, min(size_hint, 1 << 30))
    src = C.create_string_buffer(data, max(1, len(data)))
    dst = C.create_string_buffer(out_buf)
    out = bytearray()
    pos, eof = 0, False
    avail_in = C.c_size_t(0); next_in = C.c_void_p(C.addressof(src))
    avail_out = C.c_size_t(out_buf); next_out = C.c_void_p(C.addressof(dst))
    while True:
        if avail_in.value == 0 and not eof:
            n = min(chunk, len(data) - pos)
            next_in = C.c_void_p(C.addressof(src) + pos); avail_in = C.c_size_t(n)
            pos += n
            eof = n < chunk          # fread() came back short
        ok = L.BrotliEncoderCompressStream(s, 2 if eof else 0, C.byref(avail_in), C.byref(next_in),
                                           C.byref(avail_out), C.byref(next_out), None)
        assert ok == 1
        if avail_out.value == 0:
            out += dst.raw[:out_buf]
            avail_out = C.c_size_t(out_buf); next_out = C.c_void_p(C.addressof(dst))
        if L.BrotliEncoderIsFinished(s):
            out += dst.raw[:out_buf - avail_out.value]
            break
    L.BrotliEncoderDestroyInstance(s)
    return bytes(out)


def ref_stream_ops(ref, data, quality, lgwin, sizes, ops, out_buf=1 << 16, params=None):
    """Drives the reference's CompressStream with an explicit list of (size, op) calls, draining the
    output after each call the way encode.h:473 asks (repeat until no input and no more output)."""
    L = ref.lib
    L.BrotliEncoderCreateInstance.restype = C.c_void_p
    L.BrotliEncoderCreateInstance.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.BrotliEncoderSetParameter.argtypes = [C.c_void_p, C.c_int, C.c_uint32]
    L.BrotliEncoderDestroyInstance.argtypes = [C.c_void_p]
    L.BrotliEncoderHasMoreOutput.argtypes = [C.c_void_p]
    L.BrotliEncoderCompressStream.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_size_t), C.POINTER(C.c_void_p),
                                              C.POINTER(C.c_size_t), C.POINTER(C.c_void_p), C.c_void_p]
    s = L.BrotliEncoderCreateInstance(None, None, None)
    L.BrotliEncoderSetParameter(s, 1, quality)
    L.BrotliEncoderSetParameter(s, 2, lgwin)
    for k, v in (params or {}).items():        # further BrotliEncoderParameter ids (3 LGBLOCK, 4 DISABLE_LITERAL_CONTEXT_MODELING ...)
        assert L.BrotliEncoderSetParameter(s, k, v) == 1
    src = C.create_string_buffer(data, max(1, len(data)))
    dst = C.create_string_buffer(out_buf)
    out = bytearray()
    pos = 0
    for size, op in zip(sizes, ops):
        avail_in = C.c_size_t(size); next_in = C.c_void_p(C.addressof(src) + pos)
        pos += size
        while True:
            avail_out = C.c_size_t(out_buf); next_out = C.c_void_p(C.addressof(dst))
            assert L.BrotliEncoderCompressStream(s, op, C.byref(avail_in), C.byref(next_in), C.byref(avail_out),
                                                 C.byref(next_out), None) == 1
            out += dst.raw[:out_buf - avail_out.value]
            if avail_in.value == 0 and not L.BrotliEncoderHasMoreOutput(s):
                break
    L.BrotliEncoderDestroyInstance(s)
    return bytes(out)


def _digest(b):
    """Length and the first 128 bits of the SHA-256 of a byte string (or of a RefOutput standing for one)."""
    if isinstance(b, RefOutput):
        return b.digest
    return "%d:%s" % (len(b), hashlib.sha256(bytes(b)).hexdigest()[:32])


class RefOutput(object):
    """A byte string the reference produced, known by its digest: compares equal to bytes with that digest."""

    def __init__(self, digest):
        self.digest = digest

    def __len__(self):
        return int(self.digest.split(":")[0])

    def __eq__(self, other):
        if isinstance(other, (bytes, bytearray, RefOutput)):
            return _digest(other) == self.digest
        return NotImplemented

    def __repr__(self):
        return "RefOutput(%s)" % self.digest


_RECORD_PATH = os.environ.get("BROTLI_RECORD_REFERENCE")
_recorded = {}
_table = None


def _write_recorded():
    table = json.load(open(_RECORD_PATH)) if os.path.exists(_RECORD_PATH) else {}
    table.update(_recorded)
    with open(_RECORD_PATH, "w") as f:
        json.dump(table, f, indent=0, sort_keys=True)
        f.write("\n")


class RecordedRef(object):
    """The reference encoder / decoder / CLI as the suite calls them, answered from tests/golden/reference_outputs.json:
    for every call the tests make, the digest of what the unmodified reference returned (RefOutput; integers as they
    are), keyed by the call and the digests of its inputs.  The suite so compares against the reference without its
    sources or a build of them; a call that was not recorded (new arguments, or an input that drifted) fails.

    To record: build oracle/_ref (BROTLI_REFERENCE=<google/brotli checkout> python __graft_entry__.py) and run the tests
    that use this class with BROTLI_RECORD_REFERENCE=<json file>: the calls then go to the reference, the tests compare
    against its real output, and the digests are merged into that file when the process exits."""

    def __init__(self):
        global _table
        if _RECORD_PATH:
            self.live = Ref()
            if _table is None:
                _table = {}
                atexit.register(_write_recorded)
        else:
            self.live = None
            if _table is None:
                _table = json.load(open(REFERENCE_OUTPUTS))

    def _answer(self, call, inputs, run):
        key = hashlib.sha256(json.dumps([call, [_digest(x) for x in inputs]]).encode()).hexdigest()[:20]
        if self.live is not None:
            out = run(self.live)
            _recorded[key] = out if isinstance(out, int) else _digest(out)
            return out
        assert key in _table, "no recorded reference output for %r on inputs %r" % (call, [_digest(x) for x in inputs])
        v = _table[key]
        return v if isinstance(v, int) else RefOutput(v)

    def compress(self, data, quality, lgwin, mode=0):
        return self._answer(["compress", quality, lgwin, mode], [data], lambda r: r.compress(data, quality, lgwin, mode))

    def decompress(self, comp, max_out):
        return self._answer(["decompress", max_out], [comp], lambda r: r.decompress(comp, max_out))

    def max_compressed_size(self, n):
        return self._answer(["max_compressed_size", n], [], lambda r: int(r.lib.BrotliEncoderMaxCompressedSize(n)))

    def stream_ops(self, data, quality, lgwin, sizes, ops, params=None):
        """ref_stream_ops: CompressStream with an explicit list of (size, op) calls."""
        call = ["stream_ops", quality, lgwin, list(sizes), list(ops), sorted((params or {}).items())]
        return self._answer(call, [data], lambda r: ref_stream_ops(r, data, quality, lgwin, sizes, ops, params=params))

    def compress_stream(self, data, quality, lgwin, chunk):
        """cli_compress_stream: PROCESS calls of `chunk` bytes, then FINISH."""
        return self._answer(["compress_stream", quality, lgwin, chunk], [data],
                            lambda r: cli_compress_stream(r.lib, data, quality, lgwin, chunk))

    def cli(self, args, data, from_file):
        """The reference's CLI (oracle/_ref/brotli_cli_ref) run with `args` on `data` (run_cli)."""
        return self._answer(["cli", args, from_file], [data], lambda r: run_cli(REF_CLI, args, data, from_file))


def run_cli(path, args, data, from_file):
    """The CLI of c/tools/brotli.c at `path` run with `args` on `data`, read from a file (the CLI sets the size hint
    and may shrink the window from the file's length) or from a pipe; returns what it wrote."""
    if not from_file:
        return subprocess.run([path] + args + ["-c"], input=data, stdout=subprocess.PIPE, check=True).stdout
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        src, dst = os.path.join(tmp, "in"), os.path.join(tmp, "in.br")
        open(src, "wb").write(data)
        subprocess.check_call([path] + args + ["-f", "-o", dst, src])
        return open(dst, "rb").read()
