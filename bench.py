#!/usr/bin/env python3
"""
bench.py — BASELINE.json metric: corpus GB/s and merges/s through the train() merge loop.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--size-mib M] [--dump-outputs DIR]

A "step" is one merge iteration (get_stats -> arg-max with the reference tie-break -> merge) over
the whole resident token stream.  Workload at N=1: BASELINE.json configs[2], RegexTokenizer.train
(GPT-4 split pattern) on 1 GiB of synthetic UTF-8 (seed 1337), steps W..W+K of its merge loop.
With N>1 every rank holds its own 1 GiB shard (weak scaling, contiguous byte ranges of one
N GiB corpus) and the per-merge statistics delta is all-reduced over NCCL.

value   = corpus_bytes * K / t           (device-resident stream, CUDA-event time, max over ranks)
e2e     = the same through the C ABI from a pinned HOST text buffer: bpe_load_text_gpt4 (H2D of the text,
          GPT-4 split on the device, marked stream) + bpe_train(W+K merges) + D2H of the merges, wall
          clock around the calls.  Its merges must equal those of the device-resident run, which is
          loaded from the host `regex` split: a 1 GiB cross-check of the device splitter.
roofline= fused merge kernel: (4*N_in + 4*N_out bytes per launch) / CUDA-event time per launch,
          against MEASURED_PEAKS.json hbm_gbs
cpu_baseline / --impl reference = the CPU oracle port of the reference loop (oracle/bpe_oracle.c,
          base.py:13-41 + regex.py:49-63 restated in C) on a bounded sample of the same corpus.
The host regex pre-split (third-party `regex`) is outside every timed region; the e2e leg does its
own split on the device inside the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GPT4 = r"""'(?i:[sdmt]|ll|ve|re)|[^\r\n\p{L}\p{N}]?+\p{L}+|\p{N}{1,3}| ?[^\s\p{L}\p{N}]++[\r\n]*|\s*[\r\n]|\s+(?!\S)|\s+"""


def kernel_source_sha():
    """sha256 over the sources of the dominant kernel (k_merge_seg): a committed ncu capture is only quoted
    while it describes the kernel that is being timed."""
    import hashlib
    h = hashlib.sha256()
    for f in ("k_merge_seg.cuh", "k_merge.cuh", "common.cuh", "k_seg.cuh"):
        h.update(open(os.path.join(ROOT, "minbpe_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


def ncu_traffic():
    """DRAM bytes of one profiled launch of the dominant kernel (ncu --set full, committed under profiles/);
    null when no capture of the CURRENT kernel source is on record (the capture carries the source hash)."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        d = json.load(open(p))
    except Exception:  # noqa: BLE001
        return None, None
    sha = kernel_source_sha()
    if d.get("kernel_source_sha") != sha:
        return None, {"stale": True, "capture_sha": d.get("kernel_source_sha"), "current_sha": sha,
                      "note": "profiles/ncu_traffic.json was captured from another version of the kernel; re-run tools/ncu_traffic.sh"}
    return d["dram_bytes"], d


from minbpe_b200.presplit import host_cores  # noqa: E402  (affinity mask capped by the cgroup CPU quota)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# Test hook: tests/test_emu.py runs this file end to end (all legs, N = 1 and 2 ranks over gloo, tiny sizes) against the
# CPU SIMT emulator build of the library (tests/emu/), to execute the control flow of every leg in a container without a
# GPU.  Nothing below is timed meaningfully in that mode; the driver never sets the variable.
EMU = bool(os.environ.get("BPE_BENCH_EMU"))


class _HostEvent:
    def record(self, stream=None):
        self.t = time.perf_counter()

    def elapsed_time(self, other):
        return (other.t - self.t) * 1e3


def dev_sync():
    if not EMU:
        import torch
        torch.cuda.synchronize()


def new_event():
    if EMU:
        return _HostEvent()
    import torch
    return torch.cuda.Event(enable_timing=True)


def dev_tensor(values, dtype=None):
    import torch
    return torch.tensor(values, device="cpu" if EMU else "cuda", dtype=dtype)


def make_step_engine(eng, local):
    if EMU:
        sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
        from host_step import HostStepEngine
        return HostStepEngine(eng)
    from minbpe_b200.dist import GpuStepEngine
    return GpuStepEngine(eng, local)


def pin_host(arr):
    """cudaHostRegister the numpy buffer (the contract's "pinned host memory"); False if refused."""
    if EMU:
        return False
    import torch
    try:
        rc = torch.cuda.cudart().cudaHostRegister(arr.ctypes.data, arr.nbytes, 0)
        return int(rc) == 0
    except Exception:  # noqa: BLE001
        return False


def unpin_host(arr):
    import torch
    try:
        torch.cuda.cudart().cudaHostUnregister(arr.ctypes.data)
    except Exception:  # noqa: BLE001
        pass


class Watchdog:
    """The contract is ONE JSON line.  The later legs of a run (whole-loop run, cfg4, cfg5) are optional detail: if one
    of them hangs, this timer prints the line with what has been measured so far and ends the process, instead of
    leaving the driver without a number."""

    def __init__(self, seconds):
        self.line, self.timer, self.seconds = None, None, seconds

    def arm(self, line):
        self.line = line
        if self.timer is None and self.seconds > 0:
            self.timer = threading.Timer(self.seconds, self._fire)
            self.timer.daemon = True
            self.timer.start()

    def _fire(self):
        if self.line is not None:
            self.line["watchdog"] = f"a later leg did not finish within {self.seconds} s; line printed by the watchdog"
            print(json.dumps(self.line), flush=True)
        os._exit(0)

    def disarm(self):
        if self.timer is not None:
            self.timer.cancel()


def host_mem_available():
    """Bytes of host memory this process can still take: /proc/meminfo MemAvailable, capped by the cgroup's limit - usage."""
    avail = None
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable:"):
                avail = int(ln.split()[1]) * 1024
                break
    except OSError:
        pass
    for lim, cur in (("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory.current"),
                     ("/sys/fs/cgroup/memory/memory.limit_in_bytes", "/sys/fs/cgroup/memory/memory.usage_in_bytes")):
        try:
            l = open(lim).read().strip()
            if l != "max" and int(l) < (1 << 60):
                room = int(l) - int(open(cur).read().strip())
                avail = room if avail is None else min(avail, room)
        except (OSError, ValueError):
            pass
    return avail


def host_room_for(name, need_bytes, world=1):
    """None if the box has room for an optional leg's host buffers (with a 2x margin), else a {"skipped": ...} entry.
    Under torchrun rank 0 decides for everybody (the legs contain collectives)."""
    avail = host_mem_available()
    ok = 1 if (avail is None or avail >= 2 * need_bytes) else 0
    if world > 1:
        import torch
        import torch.distributed as dist
        t = dev_tensor([ok], dtype=torch.int64)
        dist.broadcast(t, src=0)
        ok = int(t.item())
    if ok:
        return None
    return {"skipped": f"{name}: needs {need_bytes / 1e9:.1f} GB of host memory for its buffers, "
                       f"{(avail or 0) / 1e9:.1f} GB available on this box (2x margin required)"}


def guarded(name, fn, *a):
    """Run an optional leg; a failure becomes {"error": ...} in the line instead of losing the whole run."""
    try:
        return fn(*a)
    except Exception as ex:  # noqa: BLE001
        import traceback
        return {"error": f"{name}: {ex!r}", "traceback": traceback.format_exc()[-1500:]}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu=0):
        self.gpu, self.rows, self.proc = gpu, [], None
        self.t_begin = self.t_end = None

    def start(self):
        """Start sampling (nvidia-smi needs ~0.2 s to produce its first line: call this well before the timed region)."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def begin(self):
        self.t_begin = time.perf_counter()

    def end(self):
        self.t_end = time.perf_counter()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([time.perf_counter()] + [x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if self.t_end is None:
            self.t_end = time.perf_counter()
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        lo = self.t_begin if self.t_begin is not None else 0.0
        rows = [r[1:] for r in self.rows if lo <= r[0] <= self.t_end + 0.03]
        window = "timed region"
        if not rows and self.rows:   # region shorter than the sampling period: the sample nearest to it
            mid = 0.5 * (lo + self.t_end)
            rows = [min(self.rows, key=lambda r: abs(r[0] - mid))[1:]]
            window = "nearest sample to the timed region"
        self.rows = rows
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


def make_corpus(size_bytes, seed):
    from minbpe_b200.presplit import chunk_offsets
    from minbpe_b200.synth import generate
    t0 = time.time()
    raw = generate(seed, size_bytes)
    t1 = time.time()
    offs = chunk_offsets(GPT4, raw)
    t2 = time.time()
    return raw, offs, {"generate_s": round(t1 - t0, 2), "presplit_s": round(t2 - t1, 2), "chunks": int(offs.size)}


# ---------------------------------------------------------------------------------------------
def cpu_port_run(raw, offs, sample_bytes, steps, warmup=0):
    """Time `steps` iterations of the oracle's C restatement of the reference loop (regex.py:49-63)
    on the first `sample_bytes` of the corpus (cut at a chunk start).  Single thread."""
    import ctypes

    import oracle
    L = oracle.lib()
    k = int(np.searchsorted(offs, sample_bytes, side="left"))
    cut = int(offs[k]) if k < offs.size else min(sample_bytes, raw.size)
    ids = raw[:cut].astype(np.int32)
    start = np.zeros(max(cut, 1), dtype=np.uint8)
    start[offs[:k].astype(np.int64)] = 1
    if cut:
        start[0] = 1
    n = ctypes.c_uint64(cut)
    pair = (ctypes.c_int32 * 2)()
    cnt = ctypes.c_int64()
    done = 0
    for i in range(warmup):
        L.orc_train_step(ids.ctypes.data, start.ctypes.data, ctypes.byref(n), 256 + i, pair, ctypes.byref(cnt))
    t0 = time.perf_counter()
    for i in range(steps):
        rc = L.orc_train_step(ids.ctypes.data, start.ctypes.data, ctypes.byref(n), 256 + warmup + i, pair, ctypes.byref(cnt))
        if rc != 0:
            break
        done += 1
    dt = time.perf_counter() - t0
    return cut, done, dt


def python_reference_run(raw, nbytes=1 << 20, merges=8):
    """The UNMODIFIED pure-Python reference (vendored to oracle/_ref by oracle/make_ref.py) on the first `nbytes`
    of the corpus: RegexTokenizer.train(text, 256 + merges) — regex.py:36-70 with its own regex split.  One core
    (the reference is single-threaded).  None when the vendored copy is absent."""
    from oracle import make_ref
    ref = make_ref.load()
    if ref is None:
        return None
    cut = nbytes
    while cut < raw.size and (raw[cut] & 0xC0) == 0x80:
        cut += 1
    text = raw[:cut].tobytes().decode("utf-8")
    tok = ref.RegexTokenizer()
    t0 = time.perf_counter()
    tok.train(text, 256 + merges)
    dt = time.perf_counter() - t0
    return {"value": cut * merges / dt / 1e9, "unit": "GB/s", "cores": 1, "kind": "reference", "merges_per_s": merges / dt,
            "seconds": dt, "first_pairs": [list(p) for p in list(tok.merges)[:4]],
            "sample": f"karpathy/minbpe RegexTokenizer.train (pure Python, incl. its regex split) on the first {cut} bytes, {merges} merges"}


def _taylorswift():
    with open(os.path.join(ROOT, "tests", "golden", "taylorswift.txt"), encoding="utf-8") as f:
        return f.read()


def cfg2_reference():
    """BASELINE configs[1] (cfg2) with the UNMODIFIED reference classes (oracle/_ref): BasicTokenizer and RegexTokenizer
    .train(taylorswift, 512), what the reference's train.py does — pure Python, one core.  None when not vendored."""
    from oracle import make_ref
    ref = make_ref.load()
    if ref is None:
        return None
    text, out = _taylorswift(), {}
    for name, cls in (("basic", ref.BasicTokenizer), ("regex", ref.RegexTokenizer)):
        tok = cls()
        t0 = time.perf_counter()
        tok.train(text, 512)
        out[name + "_seconds"] = time.perf_counter() - t0
        out[name + "_merges_sha16"] = merges_sha(np.array(list(tok.merges), dtype=np.int32))
    out["what"] = "karpathy/minbpe {Basic,Regex}Tokenizer.train(tests/taylorswift.txt, 512), unmodified pure Python, 1 core"
    return out


def cfg2_leg(device):
    """The same two calls through the product classes (minbpe_b200.BasicTokenizer / RegexTokenizer over the C ABI): text in,
    merges + vocab out, wall clock, median of 3; merges compared with the golden vectors the reference produced."""
    from minbpe_b200 import BasicTokenizer, RegexTokenizer
    text, out = _taylorswift(), {}
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "golden_train.json")))
    for name, cls in (("basic", BasicTokenizer), ("regex", RegexTokenizer)):
        tok = cls(device=device)
        tok.train(text, 300)                 # warm-up: handle, class tables, allocations
        runs = []
        for _ in range(3):
            t0 = time.perf_counter()
            tok.train(text, 512)
            runs.append(time.perf_counter() - t0)
        out[name + "_seconds"] = sorted(runs)[1]
        out[name + "_merges_sha16"] = merges_sha(np.array(list(tok.merges), dtype=np.int32))
        out[name + "_equals_reference_golden"] = [list(p) for p in tok.merges] == golden[f"taylorswift_{name}_512"]["merges"]
    out["what"] = "minbpe_b200.{Basic,Regex}Tokenizer.train(tests/golden/taylorswift.txt, 512): str in, merges + vocab out, wall clock, median of 3"
    return out


def _ref_worker(args):
    seed, shard, nbytes, steps, warmup = args
    from minbpe_b200.presplit import chunk_offsets_1proc
    from minbpe_b200.synth import generate
    import regex
    raw = generate(seed + 1000 * (shard + 1), nbytes, threads=1)
    offs = chunk_offsets_1proc(regex.compile(GPT4), raw.tobytes())
    return cpu_port_run(raw, offs, nbytes, steps, warmup)


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle C port of base.py:13-41 + regex.py:49-63) on the host
    cores this process may use (affinity mask capped by the cgroup quota): one independent replica of the merge
    loop per core, each on its own 16 MiB shard of synthetic text.  Three passes, the median is reported, with the
    parallel efficiency against one replica running alone; the pure-Python reference itself is timed beside it."""
    import multiprocessing as mp
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    oracle.build()
    cores = min(host_cores(), 64)
    shard = 16 << 20
    steps = args.steps
    warm = min(args.warmup, 1)
    t0 = time.perf_counter()
    solo = _ref_worker((args.seed, 0, shard, steps, warm))        # one replica alone: the per-core rate
    solo_rate = solo[0] * solo[1] / solo[2] / 1e9
    passes = []
    with mp.get_context("fork").Pool(cores) as pool:
        for _ in range(3):
            res = pool.map(_ref_worker, [(args.seed, s, shard, steps, warm) for s in range(cores)])
            tmax = max(r[2] for r in res)
            passes.append((sum(r[0] * r[1] for r in res) / tmax / 1e9, tmax, sum(r[1] for r in res) / tmax / cores))
    wall = time.perf_counter() - t0
    value, tmax, merges_per_s = sorted(passes)[1]
    from minbpe_b200.synth import generate
    pyref = python_reference_run(generate(args.seed, 2 << 20, threads=1))
    sample = (f"{cores} independent single-thread replicas of the oracle C port (bpe_oracle.c orc_train_step), each "
              f"{steps} merge steps on its own 16 MiB synthetic shard (seed {args.seed}+1000*(shard+1)); time = slowest replica; "
              f"median of 3 passes")
    line = {
        "impl": "reference", "metric": "train_loop_corpus_GBps", "value": value, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": tmax / steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": "RegexTokenizer.train merge loop, GPT-4 split, synthetic UTF-8 (BASELINE configs[2] shape), "
                               "bounded 16 MiB-per-core sample", "host_cores": cores, "os_cpu_count": os.cpu_count(),
                   "wall_s": round(wall, 2)},
        "merges_per_s": merges_per_s,
        "cpu_baseline": {"value": value, "unit": "GB/s", "cores": cores, "kind": "port", "sample": sample,
                         "passes_GBps": [p[0] for p in passes], "one_replica_GBps": solo_rate,
                         "parallel_efficiency": value / (solo_rate * cores), "python_reference": pyref,
                         "cfg2_reference": None if args.no_cfg2 else cfg2_reference()},
        "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def full_run(eng, raw, offs, merges, check=True):
    """BASELINE configs[2] to completion: bpe_load_text_gpt4 + bpe_train(all merges) from the host text, then every
    merge and count compared with the oracle's weighted loop over the distinct chunks of the host `regex` split
    (oracle.c_dedup_chunks + c_train(weights): same dict as regex.py:51-54 builds, tests/test_oracle.py)."""
    from minbpe_b200 import engine as E
    eng.set_option(E.OPT_KERNEL_TIMING, 0)
    dev_sync()
    t0 = time.perf_counter()
    eng.load_text_gpt4(raw)
    t_load = time.perf_counter() - t0
    pairs, counts, done = eng.train(merges)
    dev_sync()
    t_all = time.perf_counter() - t0
    tm = eng.timing()
    peak, _ = measured_peak()
    t_loop = tm["loop_ms"] / 1e3
    out = {"merges": int(done), "requested": int(merges), "seconds": t_all, "load_seconds": t_load, "loop_seconds": t_loop,
           "init_ms": tm["init_ms"], "merges_per_s": done / t_loop, "corpus_GBps": raw.size * done / t_loop / 1e9,
           "stream_GBps": 4.0 * tm["tokens_in"] / t_loop / 1e9,
           "fused_bytes_frac_of_peak": (4.0 * tm["tokens_in"] + 4.0 * tm["tokens_out"]) / t_loop / 1e9 / peak,
           "survey_8d_read_frac_of_peak": 8.0 * tm["tokens_in"] / t_loop / 1e9 / peak,
           "table_slots": int(tm["table_slots"]), "table_used": int(tm["table_used"]),
           "same_pairs": int(sum(1 for a, b in pairs.tolist() if a == b)), "final_tokens": int(eng.stream_len()),
           "gpu_launches": int(tm["kernel_launches"]), "end_to_end_corpus_MBps": raw.size / t_all / 1e6}
    if check:
        import oracle
        t0 = time.perf_counter()
        ub, uo, uw = oracle.c_dedup_chunks(raw, offs)
        wp, wc, wn = oracle.c_train(ub.astype(np.int32), uo, merges, weights=uw)
        out["oracle_seconds"] = time.perf_counter() - t0
        out["distinct_chunks"] = int(uo.size)
        out["parity_all_merges"] = bool(wn == done and np.array_equal(pairs, wp) and np.array_equal(counts, wc))
        if not out["parity_all_merges"]:
            k = min(len(pairs), len(wp))
            bad = np.flatnonzero((pairs[:k] != wp[:k]).any(axis=1) | (counts[:k] != wc[:k]))
            out["first_mismatch"] = int(bad[0]) if bad.size else k
    eng.set_option(E.OPT_KERNEL_TIMING, 1)
    return out, pairs


# ---------------------------------------------------------------------------------------------
# Shards of the synthetic corpus, the cfg4 strong-scaling leg, and the oracle check that works at 16 GiB
def corpus_shard(seed, total_bytes, rank, world, threads):
    """Bytes [lo, hi) of the `total_bytes` synthetic corpus of `seed` that belong to `rank`: equal parts whose ends
    are moved to the next letter+space point (minbpe_b200.dist.shard_byte_range — a provable chunk boundary, so the
    ranks' chunks together are exactly RegexTokenizer's split of the whole corpus).  Generated locally, block-wise."""
    from minbpe_b200.dist import shard_byte_range
    from minbpe_b200.synth import generate
    MiB = 1 << 20

    def fetch(a, b):
        fb = a // MiB
        buf = generate(seed, ((b + MiB - 1) // MiB - fb) * MiB, threads=1, first_block=fb)
        return buf[a - fb * MiB: b - fb * MiB]
    lo, hi = shard_byte_range(total_bytes, rank, world, fetch)
    fb = lo // MiB
    buf = generate(seed, ((hi + MiB - 1) // MiB - fb) * MiB, threads=threads, first_block=fb)
    return buf[lo - fb * MiB: hi - fb * MiB], lo, hi


def oracle_unique_chunks(eng, raw, workers):
    """Distinct chunks of `raw` in first-occurrence order with multiplicities, for the weighted oracle loop
    (oracle.c_dedup_chunks), at sizes where one pass is too slow: the text is cut into <= 1 GiB pieces at
    letter+space points, each piece is split (device splitter, itself pinned against `regex` by the tests and by
    the 1 GiB cross-check of every bench run) and de-duplicated on a host thread; the per-piece tables are merged
    in text order.  -> (list of chunk bytes, weights)"""
    from concurrent.futures import ThreadPoolExecutor
    import oracle
    from minbpe_b200.dist import first_safe_cut
    piece = 1 << 30
    cuts = [0]
    while raw.size - cuts[-1] > piece:
        lo = cuts[-1] + piece - (1 << 20)
        p = first_safe_cut(raw[lo: lo + (1 << 20)])
        assert p > 0
        cuts.append(lo + p)
    cuts.append(raw.size)

    def dedup(a, b, offs):
        ub, uo, uw = oracle.c_dedup_chunks(raw[a:b], offs, cap_chunks=1 << 22, cap_bytes=1 << 28)
        ends = np.append(uo[1:], ub.size).astype(np.int64)
        blob = ub.tobytes()
        return [blob[int(x):int(y)] for x, y in zip(uo.astype(np.int64), ends)], uw

    futs = []
    with ThreadPoolExecutor(max(1, workers)) as pool:
        for a, b in zip(cuts[:-1], cuts[1:]):
            offs = eng.split_gpt4(raw[a:b])
            futs.append(pool.submit(dedup, a, b, offs))
        parts = [f.result() for f in futs]
    return merge_unique(parts)


def merge_unique(parts):
    """Merge per-piece (chunks, weights) tables in text order, keeping first-occurrence order."""
    index, chunks, weights = {}, [], []
    for cs, ws in parts:
        for c, w in zip(cs, np.asarray(ws).tolist()):
            k = index.get(c)
            if k is None:
                index[c] = len(chunks)
                chunks.append(c)
                weights.append(w)
            else:
                weights[k] += w
    return chunks, weights


def oracle_train_unique(chunks, weights, merges):
    import oracle
    lens = np.fromiter(map(len, chunks), dtype=np.int64, count=len(chunks))
    offs = np.zeros(len(chunks), dtype=np.uint64)
    if len(chunks) > 1:
        offs[1:] = np.cumsum(lens[:-1])
    ids = np.frombuffer(b"".join(chunks), dtype=np.uint8).astype(np.int32)
    return oracle.c_train(ids, offs, merges, weights=np.asarray(weights, dtype=np.int64))


def merges_sha(pairs):
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(pairs, dtype=np.int32).tobytes()).hexdigest()[:16]


DUMP_BYTES = 64 << 20


def dump_outputs(path, **arrays):
    """--dump-outputs: what the timed train() call returned, one float64 `<name>.npy` per array (exact: ids are int32 and
    counts stay below 2**53), so that two builds run with the same arguments can be compared output for output.  All
    arrays have one row per merge; past DUMP_BYTES a fixed, seeded sample of rows is kept and its indices go to rows.npy."""
    os.makedirs(path, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = 8 + sum(a[:1].nbytes for a in arrays.values())
    if n * row_bytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // row_bytes, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def strong_host_bytes(args):
    """Host memory of the cfg4 leg over all ranks of the box: the corpus itself (the shards add up to it)."""
    return (args.strong_mib << 20) if args.strong_mib else (args.strong_gib << 30)


def encode_host_bytes(args):
    """Host memory of the cfg5 leg over all ranks: the text + an id buffer of up to 4 B per text byte (small tables)."""
    n = int(args.encode_gb * 1e9)
    return n + 4 * (n // 2 if args.encode_merges >= 8192 else n)


def strong_leg(args, eng, rank, world, local):
    """BASELINE configs[3] (cfg4): RegexTokenizer.train on `strong_gib` GiB of synthetic UTF-8 (seed 1338) sharded by
    byte range over the N GPUs, vocab 100000 (the per-merge statistics vector is the real 2*100000+1 counters).
    STRONG scaling: the corpus is fixed, rank r holds part r of N.  Two timed windows of K merges of the same run —
    dense early merges (W..W+K) and sparse later ones (S..S+K) — plus the sha256 of the merges so far (equal lines at
    N = 1, 2, 4, 8 <=> identical merges) and a check of the first merges against the oracle's weighted loop over the
    distinct chunks of the WHOLE corpus (gathered from all ranks).  N=1 runs the single-GPU device-driven loop
    (bpe_train), N>1 the sharded loop (--exchange: NCCL all-reduces by default, the NVLink peer-memory kernels opt-in)."""
    import torch.distributed as dist
    from minbpe_b200 import engine as E
    from minbpe_b200.dist import ShardedTrainer
    total = (args.strong_mib << 20) if args.strong_mib else (args.strong_gib << 30)
    vocab = args.strong_vocab
    M = vocab - 256
    K, W, S = args.steps, args.warmup, args.strong_sparse_at
    threads = max(1, host_cores() // world)
    t0 = time.time()
    raw, lo, hi = corpus_shard(1338, total, rank, world, threads)
    gen_s = time.time() - t0

    def sync():
        dev_sync()
        if world > 1:
            dist.barrier()
            dev_sync()

    def tmax(x):
        if world == 1:
            return x
        import torch
        t = dev_tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sync()
    t0 = time.perf_counter()
    eng.load_text_gpt4(raw)
    dev_sync()
    load_s = tmax(time.perf_counter() - t0)
    eng.set_option(E.OPT_KERNEL_TIMING, 0)
    windows = {}
    exchange_used, exchange_fallback = None, None
    if world == 1:
        eng.set_option(E.OPT_VOCAB_CAP, vocab)
        done_total, all_pairs = 0, []

        def advance(k, timed=None):
            nonlocal done_total
            if k <= 0:
                return
            dev_sync()
            p, c, d = eng.train(k, first_idx=256 + done_total)
            tm = eng.timing()
            assert d == k, "corpus ran out of pairs"
            all_pairs.append(p)
            done_total += d
            if timed:
                windows[timed] = {"first_merge": done_total - k, "merges": k, "seconds": tm["loop_ms"] / 1e3,
                                  "merges_per_s": k / (tm["loop_ms"] / 1e3), "tokens_in": int(tm["tokens_in"])}
        advance(W)
        advance(K, "dense")
        advance(S - done_total)
        advance(K, "sparse")
        pairs = np.concatenate(all_pairs)
        eng.set_option(E.OPT_VOCAB_CAP, 0)
    else:
        step = make_step_engine(eng, local)
        tr = ShardedTrainer(step, rank, world, poll_every=16, exchange=args.exchange)
        tr.prepare(M)

        def window(k, name):
            sync()
            ev0, ev1 = new_event(), new_event()
            first = tr.done
            ev0.record(step.stream)
            tr.run(k)
            ev1.record(step.stream)
            sync()
            t = tmax(ev0.elapsed_time(ev1) / 1e3)
            windows[name] = {"first_merge": first, "merges": tr.done - first, "seconds": t, "merges_per_s": (tr.done - first) / t}
        tr.run(W)
        window(K, "dense")
        tr.run(S - tr.done)
        window(K, "sparse")
        pairs, _, n = tr.result()
        pairs = pairs[:n]
        exchange_used, exchange_fallback = tr.exchange, getattr(tr, "exchange_fallback", None)
    # ---- parity: first P merges vs the oracle over the distinct chunks of the whole corpus ----
    P = min(args.strong_check, len(pairs))
    parity = None
    if P > 0:
        t0 = time.time()
        chunks, weights = oracle_unique_chunks(eng, raw, threads)
        if world > 1:
            gathered = [None] * world
            dist.all_gather_object(gathered, (chunks, weights))
            if rank == 0:
                chunks, weights = merge_unique(gathered)
        if rank == 0:
            wp, wc, wn = oracle_train_unique(chunks, weights, P)
            parity = {"merges_checked": int(P), "equal": bool(wn == P and np.array_equal(pairs[:P], wp)),
                      "distinct_chunks": len(chunks), "seconds": round(time.time() - t0, 1),
                      "how": "oracle.c_train(weights) over the distinct chunks of the whole corpus (device split of every rank's "
                             "shard, host de-duplication, tables merged in rank = text order)"}
    if world > 1:
        try:
            step.e.xchg_detach()
        except Exception:  # noqa: BLE001
            pass
        sync()
    out = {"workload": f"BASELINE configs[3]: RegexTokenizer.train, {total / (1 << 30):g} GiB synthetic UTF-8 (seed 1338), vocab {vocab}, "
                       f"{world} GPU(s), contiguous byte-range shards cut at letter+space", "scaling": "strong",
           "bytes_total": total, "bytes_this_rank": int(hi - lo), "vocab": vocab, "delta_vector_bytes": (2 * vocab + 1) * 8,
           "exchange": "none (1 GPU)" if world == 1 else (
               "NVLink peer memory kernels (k_xchg_cand on ties + k_xchg_apply), no NCCL per merge" if exchange_used == "p2p" else
               "NCCL all-reduce MIN (8 B) + SUM (delta vector) per merge, on the kernels' stream" +
               (f" (p2p was requested; fell back: {exchange_fallback})" if exchange_fallback else "")),
           "exchanged_bytes_per_merge_per_rank": 0 if world == 1 else (2 * vocab + 1) * 8 + 8,
           "generate_s": round(gen_s, 1), "load_seconds": load_s, "windows": windows,
           "merges_sha16": merges_sha(pairs), "merges_in_sha": int(len(pairs)), "parity_vs_oracle": parity}
    return out


def encode_leg(args, eng, rank, world, merges):
    """BASELINE configs[4] (cfg5): RegexTokenizer.encode_ordinary of `encode_gb` * 1e9 bytes of synthetic UTF-8 (seed 1339)
    with a trained 32k merges table, through the C ABI call a user makes (bpe_encode_text_gpt4: host text in, host ids
    out; H2D, GPT-4 split, memoised chunk encode and D2H all inside the timed region).  N GPUs = N replicas over byte-range
    shards (chunks are independent: no exchange).  Reports the end-to-end rate, the device time of the encode kernels
    against the HBM roofline (algorithmic bytes: 1 B per text byte + 4 B per id, SURVEY.md §8d), the split kernels'
    time beside it, the oracle port (and the pure-Python reference) on a slice, and bit-exactness of a slice."""
    import torch
    import torch.distributed as dist
    import oracle
    from minbpe_b200 import engine as E
    from minbpe_b200.dist import first_safe_cut
    total = max(1, int(args.encode_gb * 1e9) // (1 << 20)) * (1 << 20)
    threads = max(1, host_cores() // world)
    raw, lo, hi = corpus_shard(1339, total, rank, world, threads)
    raw = np.ascontiguousarray(raw)
    pinned = pin_host(raw)
    # ids: at most one per byte; a 32k-entry table leaves ~0.22 per byte of this corpus (room for 0.5), a small table more
    out = np.empty((raw.size // 2 if len(merges) >= 8192 else raw.size) + 1024, dtype=np.int32)
    pin_host(out)
    eng.set_option(E.OPT_KERNEL_TIMING, 0)
    wcut = min(raw.size, 64 << 20)
    if wcut < raw.size:
        wcut += max(0, first_safe_cut(raw[wcut: wcut + (1 << 20)]))
    ids = eng.encode_text_gpt4(raw[:wcut], merges, out=out)    # warm-up: tables, allocations (the memo stays warm, as for a user)
    runs = []
    for _ in range(3):
        dev_sync()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        ids = eng.encode_text_gpt4(raw, merges, out=out)
        runs.append(time.perf_counter() - t0)
    tm = eng.timing()
    t = sorted(runs)[1]
    # device time of the kernels, separately (events inside the library, one more run)
    eng.set_option(E.OPT_KERNEL_TIMING, 1)
    ids = eng.encode_text_gpt4(raw, merges, out=out)
    st = eng.encode_stats()
    split_ms = eng.timing()["init_ms"]
    eng.set_option(E.OPT_KERNEL_TIMING, 0)
    enc_s = st["kernel_us"] / 1e6
    tt = dev_tensor([t, enc_s, split_ms / 1e3, float(raw.size), float(ids.size)], dtype=torch.float64)
    if world > 1:
        mx = tt.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = tt.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        t, enc_s, split_s, nbytes, nids = float(mx[0]), float(mx[1]), float(mx[2]), float(sm[3]), float(sm[4])
    else:
        t, enc_s, split_s, nbytes, nids = t, enc_s, split_ms / 1e3, float(raw.size), float(ids.size)
    res = None
    if rank == 0:
        peak, _ = measured_peak()
        # parity + CPU baseline on a slice of rank 0's shard, cut where chunking cannot differ
        # (single-process regex: this process holds pinned host buffers and a CUDA context — no fork() from here)
        cut = min(raw.size, 16 << 20)
        if cut < raw.size:
            cut += max(0, first_safe_cut(raw[cut: cut + (1 << 20)]))
        from minbpe_b200.presplit import chunk_offsets_1proc
        import regex
        o2 = chunk_offsets_1proc(regex.compile(GPT4), raw[:cut].tobytes())
        t0 = time.perf_counter()
        want = oracle.c_encode(raw[:cut], o2, merges)
        dt = time.perf_counter() - t0
        same = bool(np.array_equal(ids[: want.size], want))
        py = None
        try:
            from oracle import make_ref
            ref = make_ref.load()
            if ref is not None:
                tokr = ref.RegexTokenizer()
                tokr.merges = {(int(a), int(b)): 256 + i for i, (a, b) in enumerate(np.asarray(merges).tolist())}
                tokr.vocab = tokr._build_vocab()
                c2 = min(raw.size, 1 << 20)
                if c2 < raw.size:
                    c2 += max(0, first_safe_cut(raw[c2: c2 + (1 << 16)]))
                txt = raw[:c2].tobytes().decode("utf-8")
                t0 = time.perf_counter(); rid = tokr.encode_ordinary(txt); pdt = time.perf_counter() - t0
                py = {"value": c2 / pdt / 1e9, "unit": "GB/s", "cores": 1, "kind": "reference", "seconds": pdt,
                      "equal_ids": bool(rid == ids[: len(rid)].tolist()),
                      "sample": f"karpathy/minbpe RegexTokenizer.encode_ordinary (pure Python) on the first {c2} bytes"}
        except Exception as ex:  # noqa: BLE001
            py = {"error": repr(ex)}
        alg = nbytes + 4.0 * nids
        res = {"workload": f"BASELINE configs[4]: RegexTokenizer.encode_ordinary, {total} bytes synthetic UTF-8 (seed 1339), "
                           f"{len(merges)} merges, {world} GPU(s) (replicas over byte-range shards)",
               "metric": "encode_text_GBps", "value": nbytes / t / 1e9, "unit": "GB/s", "seconds": t, "runs_seconds": runs,
               "bytes": nbytes, "ids": nids, "ids_per_s": nids / t,
               "e2e": {"value": nbytes / t / 1e9, "unit": "GB/s", "h2d_bytes": float(tm["h2d_bytes"]), "d2h_bytes": float(tm["d2h_bytes"]),
                       "host_buffer": "pinned (cudaHostRegister)" if pinned else "pageable",
                       "what": "bpe_encode_text_gpt4(host text -> host ids): H2D + GPT-4 split + encode + D2H, wall clock, median of 3, max over ranks"},
               "kernels": {"encode_s": enc_s, "split_s": split_s, "encode_text_GBps": nbytes / world / enc_s / 1e9 * world,
                           "what": "device time (CUDA events in the library) of k_enc_insert/distinct/direct/count/scan/write, and of the 4 split kernels; max over ranks"},
               "roofline": {"bound": "hbm", "kernel": "k_enc_* (memoised chunk encode: insert + count + write passes)", "unit": "GB/s",
                            "achieved": alg / world / enc_s / 1e9, "peak": peak, "frac": alg / world / enc_s / 1e9 / peak,
                            "algorithmic_bytes": alg, "per_unit": "1 B read per text byte + 4 B written per id"},
               "memo": {k: st[k] for k in ("memo_chunks", "pool_ids", "direct_chunks", "long_chunks", "pieces", "fallback_pieces")},
               "cpu_baseline": {"value": cut / dt / 1e9, "unit": "GB/s", "cores": 1, "kind": "port", "seconds": dt,
                                "sample": f"oracle/bpe_oracle.c orc_encode (regex.py:92-121 restated in C) on the first {cut} bytes, single thread",
                                "python_reference": py},
               "parity": {"equal": same, "ids_checked": int(want.size), "how": "ids of the first slice == oracle.c_encode(host regex split of that slice)"}}
    if pinned:
        unpin_host(raw)
        unpin_host(out)
    return res


def filtered_run_leg(eng, raw, merges, want_pairs):
    """BASELINE configs[2] to completion once more with the segment filter (BPE_OPT_SEG_FILTER = 1: from the batch after
    merges have become sparse, per-segment id signatures decide which segments a merge can touch and k_merge_seg<true> works
    through that list only).  Merges must equal those of full_run, which were checked against the oracle."""
    from minbpe_b200 import engine as E
    eng.set_option(E.OPT_KERNEL_TIMING, 0)
    eng.set_option(E.OPT_SEG_FILTER, 1)
    try:
        dev_sync()
        t0 = time.perf_counter()
        eng.load_text_gpt4(raw)
        pairs, counts, done = eng.train(merges)
        dev_sync()
        t_all = time.perf_counter() - t0
        tm = eng.timing()
    finally:
        eng.set_option(E.OPT_SEG_FILTER, 0)
        eng.set_option(E.OPT_KERNEL_TIMING, 1)
    t_loop = tm["loop_ms"] / 1e3
    return {"merges": int(done), "seconds": t_all, "loop_seconds": t_loop, "merges_per_s": done / t_loop,
            "corpus_GBps": raw.size * done / t_loop / 1e9, "gpu_launches": int(tm["kernel_launches"]),
            "filtered_segment_visits": int(tm["filter_segments"]),
            "candidate_fraction": tm["filter_candidates"] / tm["filter_segments"] if tm["filter_segments"] else None,
            "same_merges_as_full_run": bool(want_pairs is not None and done == len(want_pairs) and np.array_equal(pairs, want_pairs)),
            "what": "bpe_load_text_gpt4 + bpe_train(all merges) with BPE_OPT_SEG_FILTER = 1; candidate_fraction = share of the segments "
                    "the filtered merges had to read (the others cost an edge record and two signature words)"}


def hist_leg(eng, raw, merges, want_pairs):
    """The e2e measurement again with BPE_OPT_HIST_KERNEL = 0: at this first large stream k_hist_dense_packed (dense 16-bit counters in shared memory; never run on hardware before this round's end) is
    cross-checked and timed against k_hist_dense on the device and adopted if equal and not slower."""
    from minbpe_b200 import engine as E
    eng.set_option(E.OPT_HIST_KERNEL, 0)
    pinned = pin_host(raw)
    try:
        eng.load_text_gpt4(raw)
        eng.train(3)                       # the choice is made here (both kernels run)
        chosen = int(eng.timing()["hist_kernel"])
        runs, init = [], []
        for _ in range(3):
            dev_sync()
            t0 = time.perf_counter()
            eng.load_text_gpt4(raw)
            pairs, _, done = eng.train(merges)
            dev_sync()
            runs.append(time.perf_counter() - t0)
            init.append(eng.timing()["init_ms"])
        return {"kernel": {1: "k_hist_dense_packed", 2: "k_hist_dense"}.get(chosen, str(chosen)), "e2e_seconds": sorted(runs)[1],
                "e2e_GBps": raw.size * merges / sorted(runs)[1] / 1e9, "init_ms": sorted(init)[1],
                "same_merges": bool(done == merges and np.array_equal(pairs, want_pairs)),
                "what": "the e2e measurement of this line repeated with BPE_OPT_HIST_KERNEL = 0 (choose at the first large stream)"}
    finally:
        if pinned:
            unpin_host(raw)


def p2p_leg(eng, step, rank, world, raw, offs, W, K, want_pairs, collective_ms):
    """The timed K merges of the sharded line again with exchange = "p2p": candidate push on ties + delta pull/sum fused
    with the table update, over CUDA-IPC peer memory, no NCCL call per merge (k_xchg_cand / k_xchg_apply, bpe_step_fused).
    Set-up includes a handshake kernel; if peer memory cannot be used the ranks agree on that and the leg says why."""
    import torch.distributed as dist
    from minbpe_b200.dist import ShardedTrainer
    # the strong leg bound the engine to the stream of its own step engine: back to this one's, on which the events below
    # are recorded and torch issues the collectives of prepare()
    step.e.set_stream(step.stream.cuda_stream)
    eng.load_stream(raw, offs)
    tr = ShardedTrainer(step, rank, world, poll_every=16, exchange="p2p")
    tr.prepare(W + K)
    if tr.exchange != "p2p":
        return {"used": False, "reason": getattr(tr, "exchange_fallback", None)}
    tr.run(W)
    dev_sync(); dist.barrier(); dev_sync()
    ev0, ev1 = new_event(), new_event()
    ev0.record(step.stream)
    tr.run(K)
    ev1.record(step.stream)
    dev_sync(); dist.barrier(); dev_sync()
    t = dev_tensor([ev0.elapsed_time(ev1) / 1e3])
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    pairs, _, n = tr.result()
    same = dev_tensor([1.0 if (n == W + K and np.array_equal(pairs[: W + K], want_pairs)) else 0.0])
    dist.all_reduce(same, op=dist.ReduceOp.MIN)
    step.e.xchg_detach()
    dev_sync(); dist.barrier(); dev_sync()
    ms = float(t.item()) / K * 1e3
    return {"used": True, "ms_per_step": ms, "collective_ms_per_step": collective_ms, "same_merges_as_collective": bool(same.item() > 0.5),
            "what": "merge steps W..W+K-1 of the same shards, CUDA events on the shared stream, max over ranks"}


def merges_for_encode(eng, n_merges, train_mib=256):
    """A trained table for the encode leg when the run has none yet: RegexTokenizer.train on 256 MiB of the cfg3 corpus."""
    from minbpe_b200.synth import generate
    eng.load_text_gpt4(generate(1337, train_mib << 20))
    p, _, d = eng.train(n_merges)
    return p[:d]


def run_sharded(args, rank, world, local):
    """bench.py --gpus N>1 (one rank per GPU under torchrun).  Primary line: WEAK scaling of the cfg3-shaped loop, rank r
    holding part r of one N * size_mib corpus (parts cut at letter+space: together exactly the RegexTokenizer split of
    the whole corpus), per-merge exchanges per --exchange (default: two NCCL all-reduces on the kernels' stream; p2p =
    the NVLink peer-memory kernels of k_xchg.cuh).  `strong_cfg4` = strong_leg()."""
    import torch
    import torch.distributed as dist
    from minbpe_b200 import engine as E
    from minbpe_b200.dist import ShardedTrainer
    from minbpe_b200.presplit import chunk_offsets
    size = args.size_mib << 20
    K, W = args.steps, args.warmup
    t0 = time.time()
    threads = max(1, host_cores() // world)
    raw, lo, hi = corpus_shard(args.seed, size * world, rank, world, threads)
    offs = chunk_offsets(GPT4, raw, workers=threads)      # host `regex` split of the shard: cross-checks the device splitter
    prep_s = time.time() - t0

    if EMU:
        dist.init_process_group("gloo")
    else:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    eng = E.Engine(local)
    eng.set_option(E.OPT_KERNEL_TIMING, 1)
    eng.set_option(E.OPT_HIST_KERNEL, 2)      # iteration-0 histogram with the kernel that has run on B200s (see run_ours)
    step = make_step_engine(eng, local)
    sampler = None
    if rank == 0:
        sampler = ClockSampler(local)
        sampler.start()

    def sync_all():
        dev_sync()
        dist.barrier()
        dev_sync()

    # ---- e2e: host buffers -> merges through the C ABI (device split + sharded loop), wall clock, max over ranks ----
    pinned = pin_host(raw)
    eng.load_text_gpt4(raw)          # untimed warm-up of the load path ...
    ShardedTrainer(step, rank, world, poll_every=16, exchange=args.exchange).prepare(W + K)   # ... and of the first histogram / table build
    sync_all()
    t0 = time.perf_counter()
    eng.load_text_gpt4(raw)
    h2d = eng.timing()["h2d_bytes"]
    tr = ShardedTrainer(step, rank, world, poll_every=16, exchange=args.exchange)
    tr.prepare(W + K)
    tr.run()
    pairs_e2e, _, n_e2e = tr.result()
    sync_all()
    t_e2e = dev_tensor([time.perf_counter() - t0])
    dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)

    # ---- device-resident: W warm-up merges, then exactly K timed; stream loaded from the HOST regex split ----
    eng.load_stream(raw, offs)
    tr = ShardedTrainer(step, rank, world, poll_every=16, exchange=args.exchange)
    tr.prepare(W + K)
    tr.run(W)
    sync_all()
    if sampler:
        sampler.begin()
    ev0, ev1 = new_event(), new_event()
    eng.timing()
    ev0.record(step.stream)
    t0 = time.perf_counter()
    tr.run(K)
    ev1.record(step.stream)
    sync_all()
    wall = time.perf_counter() - t0
    if sampler:
        sampler.end()
    clocks = sampler.stop() if sampler else None
    t_loop = dev_tensor([ev0.elapsed_time(ev1) / 1e3])
    dist.all_reduce(t_loop, op=dist.ReduceOp.MAX)
    pairs, counts, n = tr.result()
    tm = eng.timing()
    ok = (n == W + K) and np.array_equal(pairs[: W + K], pairs_e2e)
    merge_ms = dev_tensor([tm["merge_kernel_ms"] / max(n, 1)])   # CUDA events around the merge launches, all W+K steps
    merge_all = [torch.zeros_like(merge_ms) for _ in range(world)]
    dist.all_gather(merge_all, merge_ms)
    line = None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, merges=pairs[W:W + K], counts=counts[W:W + K])
    if rank == 0:
        t = float(t_loop.item())
        peak, peak_src = measured_peak()
        k_ms = t / K * 1e3
        bytes_per_launch = 4.0 * (tm["tokens_in"] + tm["tokens_out"]) / max(n, 1)
        V = 256 + W + K
        line = {
            "metric": "train_loop_corpus_GBps", "value": size * world * K / t / 1e9, "unit": "GB/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": t / K * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": f"RegexTokenizer.train merge loop (GPT-4 split), {args.size_mib} MiB synthetic UTF-8 per GPU "
                                   f"(seed {args.seed}): rank r = part r of one {args.size_mib * world} MiB corpus, parts cut at "
                                   f"letter+space (a provable chunk boundary), merge steps {W}..{W + K - 1}; per merge: " + (
                                       "candidate push on ties + delta pull/sum fused with the table update, over NVLink peer memory "
                                       "(k_xchg.cuh), no NCCL call" if tr.exchange == "p2p" else
                                       "all-reduce MIN of the tie-break candidate (8 B) + all-reduce SUM of the statistics delta, NCCL "
                                       "on the stream the kernels run on"),
                       "parallelism": f"shard{world}", "prep_s": round(prep_s, 1), "consistent": bool(ok),
                       "exchange_used": tr.exchange, "exchange_fallback_reason": getattr(tr, "exchange_fallback", None),
                       "shard_bytes_rank0": int(hi - lo),
                       "l2": "per-GPU stream >> 126 MB L2, re-read from HBM every step",
                       "timing": "CUDA events on the shared stream, max over ranks, barrier + synchronize on both sides"},
            "merges_per_s": K / t, "wall_ms_per_step": wall / K * 1e3,
            "gpu_launches": int(tm["kernel_launches"]),
            "clocks": clocks,
            "phases_ms": {"step": k_ms, "merge_kernels_per_rank": [float(x.item()) for x in merge_all],
                          "select_exchange_apply": k_ms - max(float(x.item()) for x in merge_all),
                          "how": "merge = CUDA events around the merge launches (every rank); the rest of the step = arg-max, tie filter, "
                                 "first-occurrence scan, candidate exchange, delta exchange + table update, and waiting for the slowest rank"},
            "exchange": {"kind": "NVLink peer memory (CUDA IPC), hand-written kernels (k_xchg.cuh)" if tr.exchange == "p2p" else
                                 "NCCL all-reduce MIN (8 B candidate) + SUM (delta vector) per merge, issued on the kernels' stream" +
                                 (f" (p2p was requested; fell back: {tr.exchange_fallback})" if getattr(tr, "exchange_fallback", None) else ""),
                         "delta_vector_bytes": (2 * V + 1) * 8},
            "roofline": {"bound": "hbm", "kernel": "k_merge_seg (rank 0; rate over the whole step incl. exchanges)",
                         "achieved": bytes_per_launch / (k_ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": bytes_per_launch / (k_ms / 1e3) / 1e9 / peak, "traffic": None, "peak_source": peak_src, "ms_per_launch": k_ms},
            "cpu_baseline": None,
            "strong_cfg4": None, "encode_cfg5": None, "p2p_trial": None,
            "e2e": {"value": size * world * (W + K) / float(t_e2e.item()) / 1e9, "unit": "GB/s",
                    "h2d_bytes_per_step": h2d / (W + K), "d2h_bytes_per_step": 16.0, "seconds": float(t_e2e.item()),
                    "host_buffer": "pinned (cudaHostRegister)" if pinned else "pageable",
                    "what": "per rank: bpe_load_text_gpt4(host shard text: H2D + device split) + sharded loop of W+K merges + merges D2H, wall clock, max over ranks"},
            "first_pairs": pairs[W:W + 4].tolist(), "merges_sha16": merges_sha(pairs[: W + K]),
        }
    # ---- optional detail legs (every rank arms the same watchdog: a leg that hangs ends all ranks, rank 0 printing the
    #      contract line as it stands; a leg that raises on every rank is reported as {"error": ...}) ----
    dog = Watchdog(args.leg_budget_s)
    dog.arm(line)
    if pinned:
        unpin_host(raw)
    strong, enc = None, None
    if args.strong_gib > 0 or args.strong_mib > 0:
        strong = host_room_for("strong_cfg4", strong_host_bytes(args), world) or \
            guarded("strong_cfg4", strong_leg, args, eng, rank, world, local)
    if args.encode_gb > 0:
        enc = host_room_for("encode_cfg5", encode_host_bytes(args), world) or \
            guarded("encode_cfg5", lambda: encode_leg(args, eng, rank, world, merges_for_encode(eng, args.encode_merges, args.encode_train_mib)))
    # last: the same K merges once more with the per-merge exchanges done by our NVLink peer-memory kernels (k_xchg.cuh)
    # instead of the two NCCL calls — a trial: those kernels have only run on the CPU emulator (DESIGN.md §5)
    dog.disarm()
    if rank == 0:
        line["strong_cfg4"], line["encode_cfg5"] = strong, enc
    p2p = None
    if not EMU and not args.no_p2p_trial and args.exchange != "p2p":
        dog2 = Watchdog(min(120, args.leg_budget_s))     # its own, short budget: a rank that fails alone leaves the others in a collective
        dog2.arm(line)
        p2p = guarded("p2p_trial", p2p_leg, eng, step, rank, world, raw, offs, W, K, pairs[: W + K],
                      float(t_loop.item()) / K * 1e3 if rank == 0 else 0.0)
        dog2.disarm()
    if rank == 0:
        line["p2p_trial"] = p2p
        print(json.dumps(line), flush=True)
    # The line is out.  Leave without tearing NCCL and the peer mappings down: after a leg that died half-way on some rank a
    # collective in the teardown would wait for that rank until NCCL's own timeout; process exit releases everything.
    sys.stdout.flush()
    os._exit(0)


# ---------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun for --gpus > 1")
    size = args.size_mib << 20
    K, W = args.steps, args.warmup

    if world > 1 or os.environ.get("BPE_BENCH_FORCE_SHARDED"):   # the env switch runs the sharded loop on one rank (tests)
        return run_sharded(args, rank, world, local)

    # host-side preparation, before CUDA is touched (the pre-split forks worker processes)
    raw, offs, prep = make_corpus(size, args.seed)
    cpu = None
    if not args.no_cpu_baseline:
        import oracle
        oracle.build()
        sample = min(size, 64 << 20)
        cut, done, dt = cpu_port_run(raw, offs, sample, 8, 0)
        cpu = {"value": cut * done / dt / 1e9, "unit": "GB/s", "cores": 1, "kind": "port",
               "sample": f"first {cut} bytes of the same corpus, {done} merge steps of oracle/bpe_oracle.c orc_train_step "
                         f"(C restatement of base.py:13-41 + regex.py:49-63), {dt:.1f} s, single thread",
               "merges_per_s": done / dt, "python_reference": python_reference_run(raw)}

    from minbpe_b200 import engine as E
    if not EMU:
        torch.cuda.set_device(local)
    eng = E.Engine(local)
    eng.set_option(E.OPT_KERNEL_TIMING, 1)
    # the contract line is measured on kernels that have run on B200s: the iteration-0 histogram with k_hist_dense (the
    # library's default); the automatic choice (cross-check + timing of k_hist_dense_packed) is the `hist_packed` leg below
    eng.set_option(E.OPT_HIST_KERNEL, 2)

    sampler = ClockSampler(local)
    sampler.start()   # sampling runs from here; only the rows inside the timed region are reported
    # ---- e2e: C-ABI calls from host buffers (upload + device split + W+K merges + merges back) ----
    pinned = pin_host(raw)
    # untimed warm-up of the same calls (class tables, first-touch of the big device allocations, clocks)
    eng.load_text_gpt4(raw)
    eng.train(W)
    dev_sync()
    e2e_runs = []
    for _ in range(3):   # the wall clock of a 0.2 s region is noisy (allocator, PCIe): report the median run
        t0 = time.perf_counter()
        eng.load_text_gpt4(raw)
        load_tm = eng.timing()
        t_load = time.perf_counter() - t0
        pairs_e2e, _, done = eng.train(W + K)
        dev_sync()
        e2e_runs.append((time.perf_counter() - t0, t_load))
        assert done == W + K, "corpus ran out of pairs"
    tm_e2e = eng.timing()
    t_e2e, t_load = sorted(e2e_runs)[1]
    h2d = load_tm["h2d_bytes"]
    d2h = tm_e2e["d2h_bytes"]

    # ---- device-resident: W warm-up steps, then exactly K timed steps ----
    eng.load_stream(raw, offs)
    eng.train(W)
    dev_sync()
    sampler.begin()
    t0 = time.perf_counter()
    pairs, counts, done = eng.train(K, first_idx=256 + W)
    dev_sync()
    wall = time.perf_counter() - t0
    sampler.end()
    clocks = sampler.stop()
    tm = eng.timing()
    assert done == K
    assert np.array_equal(pairs, pairs_e2e[W:W + K]), "timed run and e2e run disagree"
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, merges=pairs, counts=counts)
    t_loop = tm["loop_ms"] / 1e3          # CUDA events on the library's stream, around the K iterations
    value = size * K / t_loop / 1e9
    n_in, n_out = tm["tokens_in"], tm["tokens_out"]
    peak, peak_src = measured_peak()
    k_ms = tm["merge_kernel_ms"] / K
    achieved = (4.0 * n_in + 4.0 * n_out) / K / (k_ms / 1e3) / 1e9
    line = {
        "metric": "train_loop_corpus_GBps", "value": value, "unit": "GB/s", "n_gpus": 1, "steps": K, "warmup": W,
        "ms_per_step": t_loop / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32", "data": "synthetic",
        "config": {"workload": f"BASELINE configs[2]: RegexTokenizer.train merge loop (GPT-4 split) on {args.size_mib} MiB synthetic "
                               f"UTF-8 seed {args.seed}, merge steps {W}..{W + K - 1} of 32512", "tokens_start": int(raw.size),
                   "chunks": prep["chunks"], "l2": "stream (>= 4 bytes/token, far larger than the 126 MB L2) is re-read from HBM every step",
                   "timing": "CUDA events on the library stream around the K enqueued iterations; wall-clock check in wall_ms_per_step",
                   "prep": prep},
        "merges_per_s": K / t_loop,
        "stream_GBps": 4.0 * n_in / t_loop / 1e9,
        "algorithmic_GBps_survey_8d": (8.0 * n_in + 4.0 * n_out) / t_loop / 1e9,
        "wall_ms_per_step": wall / K * 1e3,
        "gpu_launches": int(tm["kernel_launches"]),
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": "k_merge_seg (fused merge + in-place segment compaction + stats delta)",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic()[0],
                     "traffic_capture": ncu_traffic()[1],
                     "peak_source": peak_src, "bytes_per_launch": (4.0 * n_in + 4.0 * n_out) / K, "ms_per_launch": k_ms,
                     "loop_frac_in_kernel": tm["merge_kernel_ms"] / tm["loop_ms"]},
        "cpu_baseline": cpu,
        "cfg2": None, "full_run": None, "strong_cfg4": None, "encode_cfg5": None, "full_run_filtered": None, "hist_packed": None,
        "e2e": {"value": size * (W + K) / t_e2e / 1e9, "unit": "GB/s", "h2d_bytes_per_step": h2d / (W + K),
                "d2h_bytes_per_step": d2h / (W + K), "seconds": t_e2e, "merges": W + K,
                "load_seconds": t_load, "runs_seconds": [r[0] for r in e2e_runs], "host_buffer": "pinned (cudaHostRegister)" if pinned else "pageable",
                "init_ms": tm_e2e["init_ms"], "hist_kernel": "k_hist_dense",
                "what": "bpe_load_text_gpt4(host text: H2D + GPT-4 split on the device) + bpe_train(W+K) + merges D2H, wall clock, median of 3 runs"},
        "first_pairs": pairs[:4].tolist(),
    }
    # ---- optional detail legs.  The contract line above is complete; from here on a leg that fails is reported as
    #      {"error": ...} and a leg that hangs is cut off by the watchdog, which prints the line as it stands. ----
    dog = Watchdog(args.leg_budget_s)
    dog.arm(line)
    if pinned:
        unpin_host(raw)      # nothing below reads `raw` by DMA again; later legs pin their own buffers
    if not args.no_cfg2:
        line["cfg2"] = guarded("cfg2", cfg2_leg, local)
    full_pairs = None
    if args.full_merges > 0:
        r = guarded("full_run", full_run, eng, raw, offs, args.full_merges, not args.no_cpu_baseline)
        if isinstance(r, tuple):
            line["full_run"], full_pairs = r
        else:
            line["full_run"] = r
    if args.strong_gib > 0 or args.strong_mib > 0:
        line["strong_cfg4"] = host_room_for("strong_cfg4", strong_host_bytes(args)) or \
            guarded("strong_cfg4", strong_leg, args, eng, 0, 1, local)
    if args.encode_gb > 0:
        def enc():
            m = full_pairs if full_pairs is not None else merges_for_encode(eng, args.encode_merges, args.encode_train_mib)
            return encode_leg(args, eng, 0, 1, m)
        line["encode_cfg5"] = host_room_for("encode_cfg5", encode_host_bytes(args)) or guarded("encode_cfg5", enc)
    if args.full_merges > 0 and not args.no_filter_leg:
        line["full_run_filtered"] = guarded("full_run_filtered", filtered_run_leg, eng, raw, args.full_merges, full_pairs)
    if not args.no_hist_leg:
        line["hist_packed"] = guarded("hist_packed", hist_leg, eng, raw, W + K, pairs_e2e)
    dog.disarm()
    print(json.dumps(line), flush=True)
    eng.close()


def run_extras(args):
    """--extras: side measurements recorded in profiles/ (not the contract line): cfg2 wall times and
    chunk-parallel encode throughput (BASELINE configs[1] and configs[4] shapes)."""
    import torch
    from minbpe_b200 import BasicTokenizer, RegexTokenizer
    from minbpe_b200 import engine as E
    from minbpe_b200.presplit import chunk_offsets
    from minbpe_b200.synth import generate
    out = {}
    text = open(os.path.join(ROOT, "tests", "golden", "taylorswift.txt"), encoding="utf-8").read()
    for name, cls in (("basic", BasicTokenizer), ("regex", RegexTokenizer)):
        tok = cls()
        tok.train(text, 300)  # warm-up (context, allocations)
        t0 = time.perf_counter(); tok.train(text, 512); torch.cuda.synchronize(); dt = time.perf_counter() - t0
        t1 = time.perf_counter(); ids = tok.encode(text); torch.cuda.synchronize(); de = time.perf_counter() - t1
        out[f"cfg2_{name}"] = {"train_wall_s": dt, "merges_per_s": 256 / dt, "loop_ms": tok.last_timing["loop_ms"],
                               "encode_wall_s": de, "n_ids": len(ids)}
    size = args.size_mib << 20
    raw = generate(1339, size)
    offs = chunk_offsets(GPT4, raw)
    eng = E.Engine(0)
    # a longer stretch of the cfg3 loop: dense early merges, sparse later ones, pairs (a,a), re-packing
    eng.load_stream(raw, offs)
    t0 = time.perf_counter(); mp, mc, md = eng.train(1024); torch.cuda.synchronize(); dt = time.perf_counter() - t0
    tm = eng.timing()
    out["train_1024"] = {"bytes": size, "merges": int(md), "wall_s": dt, "loop_ms": tm["loop_ms"], "init_ms": tm["init_ms"],
                         "merges_per_s": md / (tm["loop_ms"] / 1e3), "tokens_in_sum": tm["tokens_in"], "tokens_out_sum": tm["tokens_out"],
                         "stream_GBps": 4.0 * tm["tokens_in"] / (tm["loop_ms"] / 1e3) / 1e9, "same_pairs": int(sum(1 for a, b in mp.tolist() if a == b)),
                         "table_slots": tm["table_slots"], "final_tokens": int(eng.stream_len())}
    # the literal two-pass loop of the north star (full pair histogram every iteration: BPE_OPT_RESCAN)
    sub = 256 << 20
    eng.load_stream(raw[:sub], offs[: int(np.searchsorted(offs, sub))])
    eng.set_option(E.OPT_RESCAN, 1); eng.set_option(E.OPT_KERNEL_TIMING, 1)
    eng.train(3)
    _, _, rd = eng.train(8, first_idx=259)
    tr = eng.timing()
    eng.set_option(E.OPT_RESCAN, 0); eng.set_option(E.OPT_KERNEL_TIMING, 0)
    hist_ms = (tr["loop_ms"] - tr["merge_kernel_ms"]) / max(rd, 1)
    out["rescan_256MiB"] = {"merges": int(rd), "loop_ms_per_merge": tr["loop_ms"] / max(rd, 1), "merge_ms": tr["merge_kernel_ms"] / max(rd, 1),
                            "hist_argmax_ms": hist_ms, "hist_GBps": 4.0 * tr["tokens_in"] / max(rd, 1) / (hist_ms / 1e3) / 1e9}
    # device-side GPT-4 splitter (SURVEY §8f N1): text bytes in, chunk offsets / marked stream out
    eng.split_gpt4(raw[: 16 << 20])  # warm-up (tables, allocations)
    eng.set_option(E.OPT_KERNEL_TIMING, 1)
    t0 = time.perf_counter(); got = eng.split_gpt4(raw); dt = time.perf_counter() - t0
    k_ms = eng.timing()["init_ms"]
    t0 = time.perf_counter(); eng.load_text_gpt4(raw); torch.cuda.synchronize(); dl = time.perf_counter() - t0
    eng.set_option(E.OPT_KERNEL_TIMING, 0)
    t0 = time.perf_counter(); eng.load_stream(raw, offs); torch.cuda.synchronize(); dh = time.perf_counter() - t0
    out["split_gpt4"] = {"bytes": size, "chunks": int(got.size), "equal_host_regex": bool(np.array_equal(got, offs)),
                         "offsets_wall_s": dt, "kernels_ms": k_ms, "kernels_GBps_text": size / (k_ms / 1e3) / 1e9,
                         "load_text_wall_s": dl, "load_stream_from_host_offsets_wall_s": dh}
    eng.load_stream(raw[: 64 << 20], offs[: int(np.searchsorted(offs, 64 << 20))])
    merges, _, done = eng.train(2048)
    torch.cuda.synchronize()
    t0 = time.perf_counter(); ids = eng.encode(raw, offs, merges); torch.cuda.synchronize(); dt = time.perf_counter() - t0
    tm = eng.timing()
    out["encode"] = {"bytes": size, "merges": int(done), "chunks": int(offs.size), "ids": int(ids.size), "wall_s": dt,
                     "GBps_e2e": size / dt / 1e9, "h2d_bytes": tm["h2d_bytes"], "d2h_bytes": tm["d2h_bytes"]}
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size-mib", type=int, default=1024, help="corpus bytes per GPU (MiB)")
    ap.add_argument("--seed", type=int, default=1337)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--full-merges", type=int, default=32512,
                    help="N=1: also run the whole train() loop (this many merges, configs[2] = 32512) from the host text "
                         "and compare every merge with the oracle; 0 = skip")
    ap.add_argument("--strong-gib", type=int, default=16,
                    help="also run BASELINE configs[3] (strong scaling: this many GiB in total over the N GPUs, vocab "
                         "--strong-vocab) and report it as strong_cfg4; 0 = skip")
    ap.add_argument("--strong-mib", type=int, default=0, help="size of the strong leg in MiB instead of --strong-gib (small runs, tests)")
    ap.add_argument("--strong-vocab", type=int, default=100000)
    ap.add_argument("--strong-sparse-at", type=int, default=1000, help="first merge of the second (sparse) timed window of the strong leg")
    ap.add_argument("--strong-check", type=int, default=256, help="merges of the strong leg compared with the oracle (0 = none)")
    ap.add_argument("--encode-gb", type=float, default=4.0,
                    help="also run BASELINE configs[4] (encode this many 1e9 bytes with a 32k merges table; N GPUs = replicas over "
                         "byte-range shards) and report it as encode_cfg5; 0 = skip")
    ap.add_argument("--encode-merges", type=int, default=32512, help="merges of the table the encode leg uses when the run has not trained one")
    ap.add_argument("--encode-train-mib", type=int, default=256, help="... trained on this many MiB of the cfg3 corpus")
    ap.add_argument("--exchange", default=os.environ.get("BPE_EXCHANGE", "collective"), choices=["collective", "p2p"],
                    help="N>1: per-merge exchange of the sharded loop. collective = two NCCL all-reduces (validated on 2/4/8 B200s); "
                         "p2p = the hand-written NVLink peer-memory kernels of k_xchg.cuh (opt-in until validated on hardware)")
    ap.add_argument("--leg-budget-s", type=int, default=600,
                    help="wall-clock budget of the optional legs (whole-loop run, cfg4, cfg5) after the contract line is complete; "
                         "when it runs out the line is printed with the legs finished so far")
    ap.add_argument("--no-hist-leg", action="store_true", help="skip the hist_packed leg (N=1)")
    ap.add_argument("--no-cfg2", action="store_true", help="skip the cfg2 leg (taylorswift, vocab 512, both tokenizers through the classes)")
    ap.add_argument("--no-p2p-trial", action="store_true", help="N>1: skip the trial of the NVLink peer-memory exchange kernels")
    ap.add_argument("--no-filter-leg", action="store_true", help="skip the full_run_filtered leg (N=1)")
    ap.add_argument("--extras", action="store_true", help="side measurements (cfg2 wall time, encode throughput)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what they returned to DIR as float64 .npy files: merges.npy (the K merged "
                         "pairs, [K, 2]) and counts.npy (their occurrence counts, [K])")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.extras or args.impl != "ours"):
        ap.error("--dump-outputs writes the outputs of the timed merge loop of --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.extras:
        run_extras(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
