#!/usr/bin/env python3
"""Batched encode on one GPU: RegexTokenizer.encode_ordinary_batch on 1 GiB of synthetic UTF-8 (seed 1339) cut into
documents at newlines, with seeded log-normal lengths (median ~2 KiB, ~1 % of at least 64 KiB), and a 32,512-merge table
trained as bench.py's encode leg trains it (256 MiB of the seed-1337 corpus).  Prints one JSON line and writes it to --out.

Each timing is the median of 3 runs after one warm-up:
  * encode_ordinary_batch(docs, flat=True) and the list-of-lists form, wall clock through the class (utf-8 encode of every
    document, the join, the device call, the result);
  * the same call at the engine (bytes in, flat ids out), and the same bytes without separators as ONE text through
    bpe_encode_text_gpt4 — the throughput ceiling (its ids differ at the document seams by design and are not compared);
  * device time of the encode kernels and of the split kernels (BPE_OPT_KERNEL_TIMING, one separate pass each);
  * the per-document loop (encode_ordinary per document) on the first 5,000 documents.
The roofline share counts 1 B per text byte + 4 B per id over a device-to-device copy peak measured in the same process.
Parity: the batch equals the loop on those 5,000 documents, and the oracle on a seeded sample.

    python tools/bench_encode_batch.py [--gib 1] [--out profiles/r4_encode_batch.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_identity():
    """card name and power limit, read-only"""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as ex:  # noqa: BLE001
        return {"error": repr(ex)}


def copy_peak_gbs():
    """device-to-device copy of 2 GiB: read + write bytes over event time, best of 5"""
    import torch
    a = torch.empty(1 << 31, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    best = 0.0
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); b.copy_(a); e1.record(); e1.synchronize()
        best = max(best, 2 * a.numel() / (e0.elapsed_time(e1) / 1e3) / 1e9)
    del a, b
    torch.cuda.empty_cache()
    return best


def cut_documents(raw, seed):
    """document ends: the first newline at or after each seeded log-normal length (median 2 KiB, P(>= 64 KiB) ~ 1 %)"""
    rng = np.random.default_rng(seed)
    sigma = np.log(32.0) / 2.3263                       # ln(64 KiB / 2 KiB) at the 99th percentile
    lens = rng.lognormal(np.log(2048.0), sigma, size=raw.size // 256 + 16)
    targets = np.cumsum(lens).astype(np.int64)
    targets = targets[targets < raw.size]
    nl = np.flatnonzero(raw == 10)
    ends = np.unique(nl[np.minimum(np.searchsorted(nl, targets), nl.size - 1)] + 1)
    ends = ends[ends < raw.size]
    return np.concatenate([[0], ends, [raw.size]]).astype(np.int64)


def med3(fn):
    runs = []
    for _ in range(3):
        t0 = time.perf_counter()
        r = fn()
        runs.append(time.perf_counter() - t0)
    return sorted(runs)[1], runs, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=1.0)
    ap.add_argument("--loop-docs", type=int, default=5000)
    ap.add_argument("--oracle-docs", type=int, default=200)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_encode_batch.json"))
    args = ap.parse_args()

    import oracle
    import regex
    from bench import merges_for_encode
    from minbpe_b200 import RegexTokenizer
    from minbpe_b200 import engine as E
    from minbpe_b200.synth import generate
    from minbpe_b200.tokenizer import GPT4_SPLIT_PATTERN

    gpu = gpu_identity()
    peak = copy_peak_gbs()
    tok = RegexTokenizer()
    eng = tok.engine
    merges = merges_for_encode(eng, 32512)
    tok.merges = {(int(a), int(b)): 256 + i for i, (a, b) in enumerate(merges.tolist())}
    tok.vocab = tok._build_vocab()
    m = tok._merge_array()

    raw = generate(1339, int(args.gib * (1 << 30)))
    bounds = cut_documents(raw, 1339)
    rb = raw.tobytes()
    docs = [rb[a:b].decode("utf-8") for a, b in zip(bounds[:-1].tolist(), bounds[1:].tolist())]
    lens = np.diff(bounds)
    joined = b"\xff".join(rb[a:b] for a, b in zip(bounds[:-1].tolist(), bounds[1:].tolist()))

    # warm-up: tables, allocations, the memo (it stays warm across calls, as for a user)
    tok.encode_ordinary_batch(docs, flat=True)
    t_flat, runs_flat, (ids, offs) = med3(lambda: tok.encode_ordinary_batch(docs, flat=True))
    t_eng, runs_eng, _ = med3(lambda: eng.encode_batch_gpt4(joined, len(docs), m))
    eng.encode_text_gpt4(raw, m)
    t_one, runs_one, one = med3(lambda: eng.encode_text_gpt4(raw, m))

    eng.set_option(E.OPT_KERNEL_TIMING, 1)
    eng.encode_batch_gpt4(joined, len(docs), m)
    st_b, split_b = eng.encode_stats(), eng.timing()["init_ms"]
    eng.encode_text_gpt4(raw, m)
    st_1, split_1 = eng.encode_stats(), eng.timing()["init_ms"]
    eng.set_option(E.OPT_KERNEL_TIMING, 0)
    enc_b, enc_1 = st_b["kernel_us"] / 1e3, st_1["kernel_us"] / 1e3

    del ids
    t_list, runs_list, lists = med3(lambda: tok.encode_ordinary_batch(docs))
    ids, offs = eng.encode_batch_gpt4(joined, len(docs), m)
    nids = int(offs[-1])

    k = min(args.loop_docs, len(docs))
    t_loop, runs_loop, loop_ids = med3(lambda: [tok.encode_ordinary(d) for d in docs[:k]])
    loop_bytes = int(bounds[k])
    same_loop = loop_ids == lists[:k]
    rnd = np.random.default_rng(7)
    sample = sorted(rnd.choice(len(docs), size=min(args.oracle_docs, len(docs)), replace=False).tolist())
    pat = regex.compile(GPT4_SPLIT_PATTERN)
    same_oracle = all(oracle.c_encode(*oracle.split_to_stream(docs[d], pat), m).tolist() == lists[d] for d in sample)
    same_flat = all(ids[offs[d]:offs[d + 1]].tolist() == lists[d] for d in sample)

    nbytes = float(raw.size)
    alg = nbytes + 4.0 * nids
    res = {
        "gpu": gpu,
        "workload": f"RegexTokenizer.encode_ordinary_batch: {raw.size} bytes synthetic UTF-8 (seed 1339) as {len(docs)} documents cut "
                    f"at newlines (log-normal lengths, seed 1339), {len(merges)} merges trained on 256 MiB (seed 1337)",
        "documents": {"n": len(docs), "median_bytes": float(np.median(lens)), "frac_ge_64KiB": float(np.mean(lens >= 65536)),
                      "max_bytes": int(lens.max()), "ids": nids},
        "batch_flat": {"seconds": t_flat, "runs": runs_flat, "GBps": nbytes / t_flat / 1e9,
                       "what": "tok.encode_ordinary_batch(docs, flat=True), wall clock"},
        "batch_lists": {"seconds": t_list, "runs": runs_list, "GBps": nbytes / t_list / 1e9,
                        "what": "tok.encode_ordinary_batch(docs) -> list of lists, wall clock"},
        "batch_engine": {"seconds": t_eng, "runs": runs_eng, "GBps": nbytes / t_eng / 1e9,
                         "what": "Engine.encode_batch_gpt4(joined bytes) -> flat ids, wall clock"},
        "one_text_engine": {"seconds": t_one, "runs": runs_one, "GBps": nbytes / t_one / 1e9,
                            "what": "the same bytes without separators as one text, Engine.encode_text_gpt4, wall clock (ceiling)"},
        "kernels_ms": {"batch_encode": enc_b, "batch_split": split_b, "one_text_encode": enc_1, "one_text_split": split_1,
                       "ratio_encode": enc_b / enc_1, "ratio_encode_plus_split": (enc_b + split_b) / (enc_1 + split_1),
                       "what": "device time (CUDA events in the library): k_enc_* kernels; split kernels incl. the separator marking"},
        "roofline": {"bound": "hbm", "algorithmic_bytes": alg, "per_unit": "1 B read per text byte + 4 B written per id",
                     "achieved_GBps": alg / (enc_b / 1e3) / 1e9, "copy_peak_GBps": peak,
                     "frac": alg / (enc_b / 1e3) / 1e9 / peak, "kernel": "batch encode kernels (k_enc_*)"},
        "loop": {"docs": k, "bytes": loop_bytes, "seconds": t_loop, "docs_per_s": k / t_loop, "MBps": loop_bytes / t_loop / 1e6,
                 "what": "[tok.encode_ordinary(d) for d in docs[:k]]"},
        "memo": {x: st_b[x] for x in ("memo_chunks", "pool_ids", "direct_chunks", "long_chunks", "pieces", "fallback_pieces")},
        "parity": {"batch_equals_loop": bool(same_loop), "loop_docs": k, "batch_equals_oracle": bool(same_oracle),
                   "oracle_docs": len(sample), "flat_equals_lists": bool(same_flat)},
    }
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    return 0 if (same_loop and same_oracle and same_flat) else 1


if __name__ == "__main__":
    sys.exit(main())
