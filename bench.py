#!/usr/bin/env python
"""bench.py -- encoder input MB/s of the Brotli hot path on B200 (BASELINE.json metric "q5/q9").

One JSON line.  The HEADLINE keys (value / e2e / roofline / cpu_baseline) are BASELINE.json configs[1]:
every rank compresses its own 100 000 000-byte enwik8-shaped text stream at quality 5, lgwin 22
(independent streams shard without a data-path collective: weak scaling; the compressed shards are
gathered to rank 0 over NCCL inside every step).  "sub_results" carries the other configs of the
metric, each with its own value / e2e / roofline / cpu_baseline / bit_exact:

  c4  200 MB Silesia-shaped binary mix, QUALITY 9, lgwin 24 -- the q9 half of the metric (one stream per
      GPU; a single stream does not shard: replicas at N > 1, SURVEY.md 8e)
  c3  1 GiB synthetic web mix, quality 5, lgwin 22, cut into N shards: rank i compresses bytes
      [i * 2^30 / N, (i + 1) * 2^30 / N) as its own stream (strong scaling, SURVEY.md 8e)
  c5  10 000 x 64 KiB independent streams (slices of the c3 mix), quality 1, lgwin 22, stream j on
      GPU j mod N (strong scaling), one device batch per rank
  c5q5  c5's streams at quality 5 (many small web payloads as device jobs; not a BASELINE config)
  q234  the headline's 100 MB text at quality 2, 3 and 4 plus 2 000 x 64 KiB web payloads at quality 2 and 4
      (SURVEY.md 8f rank 1; not a BASELINE config; N = 1 only).  The path was built after the round's last GPU
      minute, so it runs LAST and in a CHILD PROCESS with a time limit: whatever it does on its first contact with
      hardware, the headline line is printed.

Per config:  value = whole-job input MB/s, inputs resident in HBM, shards gathered to rank 0 in the step;
e2e = the same from HOST buffers: H2D of the inputs and D2H of the compressed bytes inside the timed region
(N = 1: through the reference-facing C ABI call BrotliEncoderCompress / BrotliB200CompressBatch with pinned
buffers, and again with pageable ones = "e2e_pageable"; N > 1: pinned H2D, device call, NCCL gather to rank 0,
D2H of all shards on rank 0).  Parity ("bit_exact") is checked outside the timed region against the unmodified
reference (oracle/_ref) run on the box's CPU on the same bytes, by every rank for its own shard.

  --impl reference : the reference's own CPU encoder (oracle/_ref; falls back to the oracle port) timed on
                     the host cores on the same configs; rank 0 only.
  --configs c2,c4  : subset (the headline c2 always runs).
  --steps / --warmup : timed and untimed steps of every config.
  --dump-outputs DIR : the compressed bytes of every config's last timed step as .npy files (dump_output), to compare
                     two builds output for output; the inputs are seeded and the same in every run.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

C2_BYTES, C3_BYTES, C4_BYTES = 100_000_000, 1 << 30, 200_000_000
C5_COUNT, C5_SIZE = 10_000, 65536
C5Q5_COUNT = C5_COUNT
WORKLOADS = {
    "c2": "100 MB enwik8-shaped synthetic text (tests/corpus.py synth_text, seed 20250922+rank), quality 5, lgwin 22, one stream per GPU",
    "c3": "1 GiB synthetic web mix (synth_web, seed 20250923) cut into N shards of 2^30/N bytes, quality 5, lgwin 22, shard i on GPU i",
    "c4": "200 MB Silesia-shaped binary mix (synth_binary, seed 20250924), quality 9, lgwin 24, one stream per GPU (replicas at N > 1)",
    "c5": "10 000 x 64 KiB streams (slices of the c3 mix at offsets i*104729 mod (2^30-65536)), quality 1, lgwin 22, stream j on GPU j mod N",
    "c5q5": "c5's 10 000 x 64 KiB streams at quality 5, lgwin 22 (many small web payloads; not a BASELINE config), stream j on GPU j mod N",
    "q234": "c2's 100 MB text at quality 2, 3 and 4, lgwin 22 (SURVEY 8f rank 1; not a BASELINE config), N = 1 only, run in a child "
            "process with a time limit so that this newest path cannot take the headline line with it",
}
QL = {"c2": (5, 22), "c3": (5, 22), "c4": (9, 24), "c5": (1, 22), "c5q5": (5, 22), "q234": (4, 22)}
METRIC = "encoder input MB/s (bit-exact)"
# the headline's config: identical in both arms (the driver compares them)
HEAD_CONFIG = {"workload": WORKLOADS["c2"], "quality": 5, "lgwin": 22, "input_bytes_per_gpu": C2_BYTES,
               "l2": "no L2 flush needed: every step streams the 100 MB input and a ~3.5 GB index, far beyond the 126 MB L2"}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.stop_flag = False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.rows.append(f)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------ inputs
_WEB = None


def web_mix():
    global _WEB
    if _WEB is None:
        from corpus import synth_web
        t = time.time()
        _WEB = synth_web(C3_BYTES)
        log("generated the %d-byte web mix in %.1fs" % (len(_WEB), time.time() - t))
    return _WEB


def c5_offsets():
    return [(i * 104729) % (C3_BYTES - C5_SIZE) for i in range(C5_COUNT)]


def make_stream_input(cfg, rank, world):
    from brotli_b200.shard import shard_range
    from corpus import synth_binary, synth_text
    t = time.time()
    if cfg == "c2":
        d = synth_text(C2_BYTES, seed=20250922 + rank)
    elif cfg == "c4":
        d = synth_binary(C4_BYTES)
    else:
        lo, hi = shard_range(C3_BYTES, rank, world)
        d = web_mix()[lo:hi]
    log("rank %d: %s input %d bytes ready in %.1fs" % (rank, cfg, len(d), time.time() - t))
    return d


def ref_lib():
    """The reference CPU encoder: oracle/_ref if it was built (kind "reference"), else the oracle port."""
    from brotli_libs import REF_SO, Oracle, Ref
    if os.path.exists(REF_SO):
        return "reference", Ref()
    return "port", Oracle()


def run_threads(n, fn):
    th = [threading.Thread(target=fn, args=(i,)) for i in range(n)]
    for x in th:
        x.start()
    for x in th:
        x.join()


# ------------------------------------------------------------------------------------------ reference arm
def reference_config(cfg, lib, n_gpus, steps, warmup):
    """Times the reference on the host cores for one config; returns (value MB/s, ms_per_step, cores, sample)."""
    q, w = QL[cfg]
    ncpu = os.cpu_count() or 1
    if cfg in ("c2", "c4"):
        # one stream cannot use more than one core (single-threaded per BrotliEncoderState); N replicas -> N cores
        d0 = make_stream_input(cfg, 0, 1)
        datas = [d0] * n_gpus
        cores = min(n_gpus, ncpu)
        units = len(d0) * n_gpus
        sample = "the whole %d-byte stream per step, %d stream(s) on %d core(s)" % (len(d0), n_gpus, cores)
        def step():
            run_threads(n_gpus, lambda i: lib.compress(datas[i], q, w))
    elif cfg == "c3":
        from brotli_b200.shard import shard_range
        web = web_mix()
        shards = [web[slice(*shard_range(C3_BYTES, r, n_gpus))] for r in range(n_gpus)]
        cores = min(n_gpus, ncpu)
        units = C3_BYTES
        sample = "the whole 1 GiB mix per step, %d shard(s) on %d core(s)" % (n_gpus, cores)
        def step():
            run_threads(n_gpus, lambda i: lib.compress(shards[i], q, w))
    else:
        web = web_mix()
        count = C5_COUNT if cfg == "c5" else C5Q5_COUNT
        streams = [web[o:o + C5_SIZE] for o in c5_offsets()[:count]]
        cores = ncpu
        units = count * C5_SIZE
        sample = "all %d streams per step, dealt over %d host threads (ctypes releases the GIL)" % (count, cores)
        def step():
            def work(k):
                for i in range(k, count, cores):
                    lib.compress(streams[i], q, w)
            run_threads(cores, work)
    for _ in range(warmup):
        step()
    t0 = time.time()
    for _ in range(steps):
        step()
    dt = time.time() - t0
    return units * steps / dt / 1e6, 1e3 * dt / steps, cores, sample


def run_reference(args, rank):
    if rank != 0:
        return
    kind, lib = ref_lib()
    v, ms, cores, sample = reference_config("c2", lib, args.gpus, args.steps, args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": round(v, 2), "unit": "MB/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 2), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": HEAD_CONFIG,
            "cpu_baseline": {"value": round(v, 2), "unit": "MB/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": round(v, 2), "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "host_cores": os.cpu_count(), "sub_results": {}}
    for cfg in args.configs:
        if cfg == "c2":
            continue
        if cfg == "q234":
            d0 = make_stream_input("c2", 0, 1)
            per = {}
            for q in (2, 3, 4):
                for _ in range(args.warmup):
                    lib.compress(d0, q, 22)
                t0 = time.time()
                for _ in range(args.steps):
                    lib.compress(d0, q, 22)
                dt = (time.time() - t0) / args.steps
                per["q%d" % q] = {"value": round(len(d0) / dt / 1e6, 2), "unit": "MB/s", "ms_per_step": round(1e3 * dt, 2),
                                  "steps": args.steps, "warmup": args.warmup,
                                  "e2e": {"value": round(len(d0) / dt / 1e6, 2), "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                                  "cpu_baseline": {"value": round(len(d0) / dt / 1e6, 2), "unit": "MB/s", "cores": 1, "kind": kind,
                                                   "sample": "the whole %d-byte stream per step, 1 thread" % len(d0)}}
            line["sub_results"][cfg] = {"workload": WORKLOADS[cfg], "lgwin": 22, "per_quality": per}
            continue
        v, ms, cores, sample = reference_config(cfg, lib, args.gpus, args.steps, args.warmup)
        line["sub_results"][cfg] = {"workload": WORKLOADS[cfg], "quality": QL[cfg][0], "lgwin": QL[cfg][1],
                                    "value": round(v, 2), "unit": "MB/s", "ms_per_step": round(ms, 2),
                                    "steps": args.steps, "warmup": args.warmup,
                                    "cpu_baseline": {"value": round(v, 2), "unit": "MB/s", "cores": cores, "kind": kind, "sample": sample},
                                    "e2e": {"value": round(v, 2), "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _emit(line)


# dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed ncu captures
# (profiles/): k_walk's first launch on c2, k_q1_parse on c5.  None where no capture of that config exists.
TRAFFIC_GB = {"c2": 13.35, "c5": 114.0}   # profiles/r02u_summary.md (k_walk<1>), profiles/r01i_summary.md (k_q1_parse)


_REAL_STDOUT = None


def _claim_stdout():
    """Everything any library prints on stdout (NCCL's version banner, ...) goes to stderr; the one JSON
    line is written to the real stdout by _emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def _emit(line):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


DUMP_BUDGET = 60_000_000   # bytes of sampled float32 data in all; the size arrays stay below the rest of 64 MB


def dump_sample(configs, world):
    """Bytes kept per dumped output: DUMP_BUDGET shared by the outputs of every rank (c2, one per further config, five
    for q234, which runs at N = 1 only)."""
    outputs = 1 + sum(c in configs for c in ("c4", "c3", "c5", "c5q5")) + (5 if "q234" in configs and world == 1 else 0)
    return DUMP_BUDGET // (4 * outputs * world)


def dump_output(out_dir, name, blobs, sample):
    """What one timed call returned in its last step: DIR/<name>_sizes.npy, the length of every compressed stream, and
    DIR/<name>.npy, the streams' bytes laid end to end, as float32 -- all of them up to `sample` bytes, else the bytes
    at `sample` positions drawn with a fixed seed (numpy default_rng(0), sorted), so that two builds compare
    position by position for as long as their outputs have the same length."""
    import numpy as np
    if not out_dir:
        return
    os.makedirs(out_dir, exist_ok=True)
    data = np.frombuffer(b"".join(blobs), np.uint8)
    if data.size > sample:
        data = data[np.sort(np.random.default_rng(0).choice(data.size, sample, replace=False))]
    np.save(os.path.join(out_dir, name + ".npy"), data.astype(np.float32))
    np.save(os.path.join(out_dir, name + "_sizes.npy"), np.array([len(b) for b in blobs], np.float64))


# ------------------------------------------------------------------------------------------ GPU arm
class Ctx(object):
    pass


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        v = json.load(open(p)).get("hbm_gbs")
        if v:
            return float(v), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    return 6550.0, "fallback of /opt/skills/guides/B200_PROFILING.md (MEASURED_PEAKS.json absent)"


def bench_stream(ctx, cfg, steps, warmup, extra_warm=True):
    """One single-stream config (c2, c4, or this rank's c3 shard)."""
    import torch
    import torch.distributed as dist
    import brotli_b200
    from brotli_b200.shard import ShardGather
    L, world, rank = ctx.L, ctx.world, ctx.rank
    q, w = QL[cfg]
    data = make_stream_input(cfg, rank, world)
    n = len(data)
    h_page = torch.frombuffer(bytearray(data), dtype=torch.uint8)          # pageable host copy
    h_in = h_page.pin_memory()
    d_in = h_in.cuda()
    cap = L.BrotliEncoderMaxCompressedSize(n) + 64
    d_out = torch.empty(cap, dtype=torch.uint8, device="cuda")
    h_out = torch.empty(cap, dtype=torch.uint8).pin_memory()
    gather = ShardGather(cap, "cuda") if world > 1 else None
    h_all = torch.empty((world, gather.cap), dtype=torch.uint8).pin_memory() if (world > 1 and rank == 0) else None
    res = {"sizes": None}

    def step_device():
        sz = C.c_size_t(cap)
        assert L.BrotliB200CompressDevice(q, w, n, d_in.data_ptr(), C.byref(sz), d_out.data_ptr()), "BrotliB200CompressDevice failed"
        if gather:
            gather.gather(d_out, sz.value)
        return sz.value

    def step_e2e_c_abi(hin, hout):
        sz = C.c_size_t(cap)
        assert L.BrotliEncoderCompress(q, w, 0, n, hin.data_ptr(), C.byref(sz), hout.data_ptr()), "BrotliEncoderCompress failed"
        return sz.value

    def step_e2e_multi():
        d_in.copy_(h_in, non_blocking=True)
        sz = C.c_size_t(cap)
        assert L.BrotliB200CompressDevice(q, w, n, d_in.data_ptr(), C.byref(sz), d_out.data_ptr())
        parts = gather.gather(d_out, sz.value)
        if rank == 0:
            for r, p in enumerate(parts):
                h_all[r, :p.numel()].copy_(p, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            res["sizes"] = list(gather.sizes)
        return sz.value

    for _ in range(warmup):
        step_device()
    dt, outs = ctx.timed(step_device, steps)
    st = brotli_b200.last_stats()
    out_size = outs[-1]
    if world == 1:
        if extra_warm:
            step_e2e_c_abi(h_in, h_out)
        dt_e2e, outs2 = ctx.timed(lambda: step_e2e_c_abi(h_in, h_out), steps)
        h_pout = torch.zeros(cap, dtype=torch.uint8)
        if extra_warm:
            step_e2e_c_abi(h_page, h_pout)
        dt_page, _ = ctx.timed(lambda: step_e2e_c_abi(h_page, h_pout), steps)
        got = bytes(h_out[:out_size].numpy().tobytes())
        d2h = out_size
    else:
        if extra_warm:
            step_e2e_multi()
        dt_e2e, outs2 = ctx.timed(step_e2e_multi, steps)
        dt_page = None
        h_mine = torch.empty(out_size, dtype=torch.uint8)
        h_mine.copy_(d_out[:out_size])
        got = bytes(h_mine.numpy().tobytes())
        d2h = sum(res["sizes"]) if rank == 0 else 0
    assert outs2[-1] == out_size
    dump_output(ctx.dump, cfg if world == 1 else "%s_rank%d" % (cfg, rank), [got], ctx.dump_sample)

    # ---- parity of this very run against the reference, outside the timed region: every rank checks its own shard;
    # rank 0 also checks that the gathered copies are the bytes the ranks produced
    kind, lib = ref_lib()
    t1 = time.time(); want = lib.compress(data, q, w); t_cpu = time.time() - t1
    ok = (got == want)
    if world > 1:
        digs = [None] * world
        dist.all_gather_object(digs, hashlib.sha256(got).hexdigest())
        if rank == 0:
            for r in range(world):
                ok = ok and hashlib.sha256(bytes(h_all[r, :res["sizes"][r]].numpy().tobytes())).hexdigest() == digs[r]
        flag = torch.tensor([1 if ok else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok = bool(flag.item())
    total_in = ctx.sum_over_ranks(n)
    total_out = ctx.sum_over_ranks(out_size)
    walk_ms = st["ms_walk"]
    r = {"workload": WORKLOADS[cfg], "quality": q, "lgwin": w, "steps": steps, "warmup": warmup,
         "scaling": "strong" if cfg == "c3" else "weak",
         "input_bytes": total_in, "compressed_bytes": total_out, "bit_exact": ok,
         "value": round(total_in * steps / dt / 1e6, 2), "unit": "MB/s", "ms_per_step": round(1e3 * dt / steps, 2),
         "e2e": {"value": round(total_in * steps / dt_e2e / 1e6, 2), "unit": "MB/s",
                 "h2d_bytes_per_step": total_in, "d2h_bytes_per_step": d2h if world > 1 else out_size,
                 "path": "BrotliEncoderCompress(host in, host out), pinned buffers" if world == 1 else
                         "pinned H2D + BrotliB200CompressDevice + NCCL gather to rank 0 + D2H of all shards on rank 0"},
         "stages_ms": {k: round(st[k], 2) for k in ("ms_total", "ms_index", "ms_lz77", "ms_entropy", "ms_assemble", "ms_walk", "ms_encode")},
         "lz77": {"walk_launches": int(st["lz77_iterations"]), "chunk_walks": int(st["block_runs"]), "chunks": int(st["blocks"]),
                  "metablocks": int(st["metablocks"])},
         "gpu_launches": int(st["launches"]) * steps}
    if dt_page is not None:
        r["e2e_pageable"] = {"value": round(total_in * steps / dt_page / 1e6, 2), "unit": "MB/s",
                             "path": "BrotliEncoderCompress with pageable (malloc) host buffers, as a drop-in caller passes them"}
    # roofline of the dominant kernel, k_walk: algorithmic bytes (SURVEY.md 8d: 1 byte read + 1/ratio written per input
    # byte) of the chunks its launches walked / their summed duration (CUDA events on the job's stream)
    peak, src = hbm_peak()
    if walk_ms > 0:
        algo = st["walk_bytes"] * (1.0 + out_size / float(n))
        ach = algo / (walk_ms / 1e3) / 1e9
        r["roofline"] = {"bound": "hbm", "kernel": "k_walk", "achieved": round(ach, 3), "peak": peak, "unit": "GB/s",
                         "frac": round(ach / peak, 6), "traffic": TRAFFIC_GB.get(cfg),
                         "traffic_unit": "GB of DRAM read+write per launch (ncu --set full, profiles/)",
                         "algorithmic_gb": round(algo / 1e9, 4), "kernel_ms": round(walk_ms, 2),
                         "launches": int(st["walk_launches"]), "peak_source": src}
    if world == 1:
        r["cpu_baseline"] = {"value": round(n / t_cpu / 1e6, 2), "unit": "MB/s", "cores": 1, "kind": kind,
                             "sample": "the whole %d-byte stream once, 1 thread (the reference encoder is single-threaded per stream)" % n}
    del d_in, d_out, h_in, h_out
    torch.cuda.empty_cache()
    return r


def bench_c5(ctx, steps, warmup):
    """10 000 x 64 KiB at quality 1: stream j on GPU j mod N, one device batch per rank."""
    import numpy as np
    import torch
    import torch.distributed as dist
    import brotli_b200
    from brotli_b200.shard import ShardGather, streams_of_rank
    L, world, rank = ctx.L, ctx.world, ctx.rank
    q, w = QL["c5"]
    web = web_mix()
    offs = c5_offsets()
    mine = streams_of_rank(C5_COUNT, rank, world)
    cnt = len(mine)
    packed = np.empty(cnt * C5_SIZE, np.uint8)
    for k, j in enumerate(mine):
        packed[k * C5_SIZE:(k + 1) * C5_SIZE] = np.frombuffer(web, np.uint8, C5_SIZE, offs[j])
    h_in = torch.from_numpy(packed).pin_memory()
    d_in = h_in.cuda()
    nbytes = cnt * C5_SIZE
    cap = nbytes + 64 * cnt + 4096
    d_out = torch.empty(cap, dtype=torch.uint8, device="cuda")
    in_off = (C.c_uint64 * cnt)(*[k * C5_SIZE for k in range(cnt)])
    in_sz = (C.c_size_t * cnt)(*([C5_SIZE] * cnt))
    out_off = (C.c_uint64 * (cnt + 1))()
    out_sz = (C.c_size_t * cnt)()
    gather = ShardGather(cap, "cuda") if world > 1 else None
    h_all = torch.empty((world, gather.cap if gather else cap), dtype=torch.uint8).pin_memory() if rank == 0 else None
    kern_ms = [0.0]
    res = {}

    def step_device():
        good = L.BrotliB200CompressBatchDevice(q, w, cnt, d_in.data_ptr(), in_off, in_sz, d_out.data_ptr(), cap, out_off, out_sz)
        assert good == cnt, "BrotliB200CompressBatchDevice: %d of %d" % (good, cnt)
        dense = int(out_off[cnt])
        if gather:
            gather.gather(d_out, dense)
        return dense

    def step_e2e():
        d_in.copy_(h_in, non_blocking=True)
        dense = step_device_nogather()
        if gather:
            parts = gather.gather(d_out, dense)
        else:
            parts = [d_out[:dense]]
        if rank == 0:
            for r, p in enumerate(parts):
                h_all[r, :p.numel()].copy_(p, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            res["sizes"] = [int(p.numel()) for p in parts]
        return dense

    def step_device_nogather():
        good = L.BrotliB200CompressBatchDevice(q, w, cnt, d_in.data_ptr(), in_off, in_sz, d_out.data_ptr(), cap, out_off, out_sz)
        assert good == cnt
        return int(out_off[cnt])

    for _ in range(warmup):
        step_device()
    dt, outs = ctx.timed(step_device, steps)
    st = brotli_b200.last_stats_q1()
    dense = outs[-1]
    step_e2e()
    dt_e2e, _ = ctx.timed(step_e2e, steps)
    out_total = sum(int(out_sz[k]) for k in range(cnt))
    # the reference-facing host batch call (pageable per-stream buffers, as a caller passes them)
    streams = [web[offs[j]:offs[j] + C5_SIZE] for j in mine]
    t0 = time.time(); got = brotli_b200.compress_batch(streams, q, w, threads=16); t_host_call = time.time() - t0
    # parity: every stream of this rank against the reference; rank 0's device copy against the host-call bytes
    kind, lib = ref_lib()
    ncpu = max(1, (os.cpu_count() or 1) // world)
    want = [None] * cnt
    t1 = time.time()
    def work(k):
        for i in range(k, cnt, ncpu):
            want[i] = lib.compress(streams[i], q, w)
    run_threads(ncpu, work)
    t_cpu_all = time.time() - t1
    ok = all(a == b for a, b in zip(got, want))
    h_dense = torch.empty(dense, dtype=torch.uint8); h_dense.copy_(d_out[:dense])
    hd = h_dense.numpy()
    dump_output(ctx.dump, "c5" if world == 1 else "c5_rank%d" % rank,
                [hd[int(out_off[k]):int(out_off[k]) + int(out_sz[k])].tobytes() for k in range(cnt)], ctx.dump_sample)
    ok = ok and all(bytes(hd[int(out_off[k]):int(out_off[k]) + int(out_sz[k])].tobytes()) == want[k] for k in range(cnt))
    if world > 1:
        flag = torch.tensor([1 if ok else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok = bool(flag.item())
    total_in = ctx.sum_over_ranks(nbytes)
    total_out = ctx.sum_over_ranks(out_total)
    peak, src = hbm_peak()
    parse_ms = st["ms_parse"]
    algo = nbytes + out_total
    ach = algo / (parse_ms / 1e3) / 1e9 if parse_ms > 0 else 0.0
    r = {"workload": WORKLOADS["c5"], "quality": q, "lgwin": w, "steps": steps, "warmup": warmup, "scaling": "strong",
         "streams": C5_COUNT, "input_bytes": total_in, "compressed_bytes": total_out, "bit_exact": ok,
         "value": round(total_in * steps / dt / 1e6, 2), "unit": "MB/s", "ms_per_step": round(1e3 * dt / steps, 2),
         "e2e": {"value": round(total_in * steps / dt_e2e / 1e6, 2), "unit": "MB/s", "h2d_bytes_per_step": total_in,
                 "d2h_bytes_per_step": sum(res["sizes"]) if rank == 0 else 0,
                 "path": "pinned H2D of the packed streams + BrotliB200CompressBatchDevice + NCCL gather to rank 0 + D2H on rank 0"},
         "e2e_pageable": {"value": round(nbytes * world / t_host_call / 1e6, 2), "unit": "MB/s",
                          "path": "BrotliB200CompressBatch(host pointer arrays, pageable per-stream buffers) incl. ctypes marshalling, one call per rank"},
         "stages_ms": {k: round(st[k], 2) for k in ("ms_total", "ms_h2d", "ms_parse", "ms_code", "ms_pack", "ms_d2h")},
         "roofline": {"bound": "hbm", "kernel": "k_q1_parse", "achieved": round(ach, 3), "peak": peak, "unit": "GB/s",
                      "frac": round(ach / peak, 6), "traffic": TRAFFIC_GB.get("c5") if world == 1 else None,
                      "traffic_unit": "GB of DRAM read+write per launch (ncu --set full, profiles/)",
                      "algorithmic_gb": round(algo / 1e9, 4), "kernel_ms": round(parse_ms, 2), "launches": 1, "peak_source": src},
         "gpu_launches": int(st["launches"]) * steps}
    if world == 1:
        r["cpu_baseline"] = {"value": round(nbytes / t_cpu_all / 1e6, 2), "unit": "MB/s", "cores": ncpu, "kind": kind,
                             "sample": "all 10 000 streams once, dealt over %d host threads" % ncpu}
    return r


def bench_c5q5(ctx, steps, warmup):
    """10 000 x 64 KiB at quality 5 through BrotliB200CompressBatch (host buffers in and out: the call IS the end-to-end
    path): the streams of a rank run as device jobs of at most 128 MiB / 8 192 streams (br_api.cc compress_stream_group)."""
    import brotli_b200
    from brotli_b200.shard import streams_of_rank
    L, world, rank = ctx.L, ctx.world, ctx.rank
    q, w = QL["c5q5"]
    web = web_mix()
    offs = c5_offsets()
    mine = streams_of_rank(C5Q5_COUNT, rank, world)
    cnt = len(mine)
    streams = [web[offs[j]:offs[j] + C5_SIZE] for j in mine]
    bufs = [C.create_string_buffer(x, len(x)) for x in streams]
    sizes = (C.c_size_t * cnt)(*[len(x) for x in streams])
    caps = [L.BrotliEncoderMaxCompressedSize(len(x)) + 16 for x in streams]
    outs = [C.create_string_buffer(c) for c in caps]
    in_ptrs = (C.c_void_p * cnt)(*[C.addressof(b) for b in bufs])
    out_ptrs = (C.c_void_p * cnt)(*[C.addressof(b) for b in outs])
    caps_arr = (C.c_size_t * cnt)(*caps)
    out_sizes = (C.c_size_t * cnt)()
    nbytes = cnt * C5_SIZE

    def step():
        C.memmove(out_sizes, caps_arr, C.sizeof(caps_arr))      # capacity in, size out
        good = L.BrotliB200CompressBatch(q, w, cnt, in_ptrs, sizes, out_ptrs, out_sizes, 16)
        assert good == cnt, "BrotliB200CompressBatch: %d of %d" % (good, cnt)

    for _ in range(warmup):
        step()
    dt, _ = ctx.timed(step, steps)
    st = brotli_b200.last_stats()
    out_total = sum(out_sizes[k] for k in range(cnt))
    dump_output(ctx.dump, "c5q5" if world == 1 else "c5q5_rank%d" % rank, [outs[k].raw[:out_sizes[k]] for k in range(cnt)],
                ctx.dump_sample)
    kind, lib = ref_lib()
    ncpu = max(1, (os.cpu_count() or 1) // world)
    want = [None] * cnt
    t1 = time.time()
    def work(k):
        for i in range(k, cnt, ncpu):
            want[i] = lib.compress(streams[i], q, w)
    run_threads(ncpu, work)
    t_cpu = time.time() - t1
    ok = all(outs[k].raw[:out_sizes[k]] == want[k] for k in range(cnt))
    if world > 1:
        import torch
        import torch.distributed as dist
        flag = torch.tensor([1 if ok else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok = bool(flag.item())
    total_in = ctx.sum_over_ranks(nbytes)
    total_out = ctx.sum_over_ranks(out_total)
    v = round(total_in * steps / dt / 1e6, 2)
    r = {"workload": WORKLOADS["c5q5"], "quality": q, "lgwin": w, "steps": steps, "warmup": warmup, "scaling": "strong",
         "streams": C5Q5_COUNT, "input_bytes": total_in, "compressed_bytes": total_out, "bit_exact": ok,
         "value": v, "unit": "MB/s", "ms_per_step": round(1e3 * dt / steps, 2),
         "value_note": "host buffers in and out (pageable): value == e2e for this call",
         "e2e": {"value": v, "unit": "MB/s", "h2d_bytes_per_step": total_in, "d2h_bytes_per_step": total_out,
                 "path": "BrotliB200CompressBatch(host pointer arrays): per group of <= 128 MiB: concat into pinned memory, H2D, one device job, D2H, split"},
         "last_group_stages_ms": {k: round(st[k], 2) for k in ("ms_total", "ms_index", "ms_lz77", "ms_walk", "ms_entropy", "ms_assemble")},
         "last_group_lz77": {"walk_launches": int(st["walk_launches"]), "chunk_walks": int(st["block_runs"]), "chunks": int(st["blocks"])},
         "gpu_launches": int(st["launches"]) * steps * max(1, -(-nbytes // (128 << 20)))}
    if world == 1:
        r["cpu_baseline"] = {"value": round(nbytes / t_cpu / 1e6, 2), "unit": "MB/s", "cores": ncpu, "kind": kind,
                             "sample": "all %d streams once, dealt over %d host threads" % (cnt, ncpu)}
    return r


def q234_child(steps, warmup, dump, sample):
    """Child process of the q234 sub-result: C2's input at quality 2, 3, 4 on cuda:0; prints one JSON object."""
    import torch
    import brotli_b200
    from corpus import synth_text
    L = brotli_b200.lib()
    torch.cuda.set_device(0)
    data = synth_text(C2_BYTES, seed=20250922)
    n = len(data)
    h_in = torch.frombuffer(bytearray(data), dtype=torch.uint8).pin_memory()
    d_in = h_in.cuda()
    cap = L.BrotliEncoderMaxCompressedSize(n) + 64
    d_out = torch.empty(cap, dtype=torch.uint8, device="cuda")
    h_out = torch.empty(cap, dtype=torch.uint8).pin_memory()
    kind, lib = ref_lib()
    peak, src = hbm_peak()
    per = {}
    for q in (2, 3, 4):
      try:
        def dev():
            sz = C.c_size_t(cap)
            assert L.BrotliB200CompressDevice(q, 22, n, d_in.data_ptr(), C.byref(sz), d_out.data_ptr()), "BrotliB200CompressDevice failed"
            return sz.value
        def e2e():
            sz = C.c_size_t(cap)
            assert L.BrotliEncoderCompress(q, 22, 0, n, h_in.data_ptr(), C.byref(sz), h_out.data_ptr()), "BrotliEncoderCompress failed"
            return sz.value
        for _ in range(warmup):
            dev()
        torch.cuda.synchronize(); t0 = time.perf_counter()
        for _ in range(steps):
            out_size = dev()
        torch.cuda.synchronize(); dt = time.perf_counter() - t0
        st = brotli_b200.last_stats()
        e2e()
        torch.cuda.synchronize(); t0 = time.perf_counter()
        for _ in range(steps):
            assert e2e() == out_size
        torch.cuda.synchronize(); dt2 = time.perf_counter() - t0
        got = bytes(h_out[:out_size].numpy().tobytes())
        dump_output(dump, "q234_q%d" % q, [got], sample)
        t1 = time.time(); want = lib.compress(data, q, 22); t_cpu = time.time() - t1
        r = {"quality": q, "lgwin": 22, "steps": steps, "warmup": warmup, "input_bytes": n, "compressed_bytes": out_size,
             "bit_exact": got == want, "value": round(n * steps / dt / 1e6, 2), "unit": "MB/s", "ms_per_step": round(1e3 * dt / steps, 2),
             "e2e": {"value": round(n * steps / dt2 / 1e6, 2), "unit": "MB/s", "h2d_bytes_per_step": n, "d2h_bytes_per_step": out_size,
                     "path": "BrotliEncoderCompress(host in, host out), pinned buffers"},
             "stages_ms": {k: round(st[k], 2) for k in ("ms_total", "ms_index", "ms_lz77", "ms_entropy", "ms_assemble", "ms_walk", "ms_encode")},
             "lz77": {"walk_launches": int(st["lz77_iterations"]), "chunk_walks": int(st["block_runs"]), "chunks": int(st["blocks"]),
                      "metablocks": int(st["metablocks"])},
             "gpu_launches": int(st["launches"]) * steps,
             "cpu_baseline": {"value": round(n / t_cpu / 1e6, 2), "unit": "MB/s", "cores": 1, "kind": kind,
                              "sample": "the whole %d-byte stream once, 1 thread" % n}}
        if st["ms_walk"] > 0:
            algo = st["walk_bytes"] * (1.0 + out_size / float(n))
            ach = algo / (st["ms_walk"] / 1e3) / 1e9
            r["roofline"] = {"bound": "hbm", "kernel": "k_walk<0>", "achieved": round(ach, 3), "peak": peak, "unit": "GB/s",
                             "frac": round(ach / peak, 6), "traffic": None, "algorithmic_gb": round(algo / 1e9, 4),
                             "kernel_ms": round(st["ms_walk"], 2), "launches": int(st["walk_launches"]), "peak_source": src}
        per["q%d" % q] = r
        log("q234 child: quality %d: %s MB/s, bit_exact %s" % (q, r["value"], r["bit_exact"]))
      except Exception as e:      # (one quality failing must not hide the others)
        per["q%d" % q] = {"quality": q, "error": repr(e)}
        log("q234 child: quality %d failed: %r" % (q, e))
    result = {"workload": WORKLOADS["q234"], "lgwin": 22, "per_quality": per}
    try:      # many small streams at quality 2 and 4: 2 000 x 64 KiB web payloads as device jobs of <= 128 MiB (host buffers in and out)
        from corpus import synth_web
        cnt = 2000
        web = synth_web(cnt * C5_SIZE, 20250923)
        streams = [web[i * C5_SIZE:(i + 1) * C5_SIZE] for i in range(cnt)]
        bufs = [C.create_string_buffer(x, len(x)) for x in streams]
        sizes = (C.c_size_t * cnt)(*[len(x) for x in streams])
        caps = [L.BrotliEncoderMaxCompressedSize(len(x)) + 16 for x in streams]
        outs = [C.create_string_buffer(c) for c in caps]
        in_ptrs = (C.c_void_p * cnt)(*[C.addressof(b) for b in bufs])
        out_ptrs = (C.c_void_p * cnt)(*[C.addressof(b) for b in outs])
        caps_arr = (C.c_size_t * cnt)(*caps)
        out_sizes = (C.c_size_t * cnt)()
        ncpu = os.cpu_count() or 1
        batch = {}
        for q in (2, 4):
            def step():
                C.memmove(out_sizes, caps_arr, C.sizeof(caps_arr))
                good = L.BrotliB200CompressBatch(q, 22, cnt, in_ptrs, sizes, out_ptrs, out_sizes, 16)
                assert good == cnt, "BrotliB200CompressBatch: %d of %d" % (good, cnt)
            for _ in range(warmup):
                step()
            torch.cuda.synchronize(); t0 = time.perf_counter()
            for _ in range(steps):
                step()
            torch.cuda.synchronize(); dt = time.perf_counter() - t0
            st = brotli_b200.last_stats()
            dump_output(dump, "q234_batch_q%d" % q, [outs[k].raw[:out_sizes[k]] for k in range(cnt)], sample)
            want = [None] * cnt
            t1 = time.time()
            def work(k):
                for i in range(k, cnt, ncpu):
                    want[i] = lib.compress(streams[i], q, 22)
            run_threads(ncpu, work)
            t_cpu = time.time() - t1
            v = round(cnt * C5_SIZE * steps / dt / 1e6, 2)
            batch["q%d" % q] = {"streams": cnt, "stream_bytes": C5_SIZE, "quality": q, "lgwin": 22, "steps": steps, "warmup": warmup,
                                "bit_exact": all(outs[k].raw[:out_sizes[k]] == want[k] for k in range(cnt)),
                                "value": v, "unit": "MB/s", "ms_per_step": round(1e3 * dt / steps, 2),
                                "e2e": {"value": v, "unit": "MB/s", "h2d_bytes_per_step": cnt * C5_SIZE,
                                        "d2h_bytes_per_step": sum(out_sizes[k] for k in range(cnt)),
                                        "path": "BrotliB200CompressBatch(host pointer arrays): value == e2e for this call"},
                                "lz77": {"walk_launches": int(st["walk_launches"]), "chunk_walks": int(st["block_runs"]), "chunks": int(st["blocks"])},
                                "cpu_baseline": {"value": round(cnt * C5_SIZE / t_cpu / 1e6, 2), "unit": "MB/s", "cores": ncpu, "kind": kind,
                                                 "sample": "all %d streams once, dealt over %d host threads" % (cnt, ncpu)}}
            log("q234 child: batch quality %d: %s MB/s, bit_exact %s" % (q, v, batch["q%d" % q]["bit_exact"]))
        result["batch_2000x64KiB"] = batch
    except Exception as e:
        result["batch_2000x64KiB"] = {"error": repr(e)}
    sys.stdout.write(json.dumps(result) + "\n")
    sys.stdout.flush()


def bench_q234(steps, warmup, dump, sample):
    """Runs q234_child in a process of its own (time limit 5 minutes and 20 s per step; it needs about two minutes at 3
    steps): a crash or a hang of the newest path ends the child, not the bench."""
    cmd = [sys.executable, os.path.abspath(__file__), "--q234-child", "--steps", str(steps), "--warmup", str(warmup)]
    if dump:
        cmd += ["--dump-outputs", dump, "--dump-sample", str(sample)]
    p = subprocess.run(cmd, stdout=subprocess.PIPE, timeout=300 + 20 * (steps + warmup))
    lines = [l for l in p.stdout.decode("utf-8", "replace").splitlines() if l.startswith("{")]
    if p.returncode != 0 or not lines:
        raise RuntimeError("q234 child exited with %d" % p.returncode)
    return json.loads(lines[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps of every config")
    ap.add_argument("--warmup", type=int, default=3, help="untimed steps in front of them")
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--configs", default="c2,c4,c3,c5,c5q5,q234")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the compressed bytes of every config's last timed step "
                    "under DIR (dump_output)")
    ap.add_argument("--q234-child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--dump-sample", type=int, default=0, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.q234_child:
        q234_child(args.steps, args.warmup, args.dump_outputs, args.dump_sample)
        return
    _claim_stdout()
    args.configs = [c for c in args.configs.split(",") if c in WORKLOADS]
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    import brotli_b200
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: brotli_b200 has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = Ctx()
    ctx.L, ctx.rank, ctx.world, ctx.dump = brotli_b200.lib(), rank, world, args.dump_outputs
    ctx.dump_sample = dump_sample(args.configs, world)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """barrier + synchronize on both sides; max over ranks."""
        barrier()
        t0 = time.perf_counter()
        outs = [fn() for _ in range(steps)]
        barrier()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        return dt, outs

    def sum_over_ranks(v):
        if world == 1:
            return int(v)
        t = torch.tensor([int(v)], dtype=torch.int64, device="cuda")
        dist.all_reduce(t)
        return int(t.item())

    ctx.timed, ctx.sum_over_ranks = timed, sum_over_ranks
    sampler = ClockSampler(local_rank)
    sampler.start()
    head = bench_stream(ctx, "c2", args.steps, args.warmup)
    sampler.stop_flag = True
    sub = {}
    for cfg in args.configs:
        t0 = time.time()
        try:
            if cfg in ("c4", "c3"):
                sub[cfg] = bench_stream(ctx, cfg, args.steps, args.warmup, extra_warm=False)
            elif cfg == "c5":
                sub[cfg] = bench_c5(ctx, args.steps, args.warmup)
            elif cfg == "c5q5":
                sub[cfg] = bench_c5q5(ctx, args.steps, args.warmup)
            elif cfg == "q234" and world == 1:
                sub[cfg] = bench_q234(args.steps, args.warmup, args.dump_outputs, ctx.dump_sample)
        except Exception as e:      # a sub-result must not take the headline line with it (one rank: the others would hang)
            if world > 1:
                raise
            sub[cfg] = {"workload": WORKLOADS[cfg], "error": repr(e)}
        if cfg in sub:
            log("rank %d: %s done in %.1fs" % (rank, cfg, time.time() - t0))
    if rank == 0:
        line = {"metric": METRIC, "value": head["value"], "unit": "MB/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": HEAD_CONFIG, "bit_exact_vs_reference": head["bit_exact"], "compressed_bytes": head["compressed_bytes"],
                "clocks": sampler.summary(), "e2e": head["e2e"], "gpu_launches": head["gpu_launches"],
                "roofline": head.get("roofline"), "cpu_baseline": head.get("cpu_baseline"),
                "stages_ms": head["stages_ms"], "lz77": head["lz77"], "host_cores": os.cpu_count(),
                "sub_results": sub}
        if "e2e_pageable" in head:
            line["e2e_pageable"] = head["e2e_pageable"]
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
