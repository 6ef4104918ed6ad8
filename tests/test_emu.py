"""CPU: the kernel SOURCES of minbpe_b200/csrc on the SIMT emulator (tests/emu/, test infrastructure).

tests/emu/build_emu.py compiles b200bpe.cu — kernels and host side — with g++ against tests/emu/cuda_emu.h (one fiber
per CUDA thread, rendezvous barriers and warp collectives, guarded allocations) into libb200bpe_emu.so, which exports
the C ABI of include/b200bpe.h.  The GPU parity tests are then run against THAT library (BPE_LIB_PATH) in
subprocesses: the same test code, the same oracle, the kernels' logic executed on the CPU.

It is a logic check for a container without a GPU, NOT a product path (nothing in minbpe_b200/ loads the emulator
build) and not a substitute for `-m gpu` on a B200: performance, the PTX paths (TMA / mbarrier are emulated as
immediate copies) and the cross-GPU memory model are out of its reach.

bench.py itself is executed the same way (BPE_BENCH_EMU=1: gloo instead of NCCL, host tensors, tiny sizes), N = 1 and
N = 2 ranks under torchrun, every leg: contract line, whole-loop run, cfg4 strong leg, cfg5 encode leg — so that the
control flow the driver will run at round end has been executed at least once, with its parity checks green.

The jobs start together (they are independent processes) and each test waits for its own job."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "emu")


def _free_port():
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _env(lib):
    env = dict(os.environ)
    env.update(BPE_LIB_PATH=lib, BPE_TEST_SMALL="1", EMU_SMS="2", PYTHONDONTWRITEBYTECODE="1")
    env.pop("PYTEST_CURRENT_TEST", None)
    return env


def _pytest(lib, files, k=None, order=None, par=None):
    cmd = [sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", "-p", "no:cacheprovider", "-o", "timeout=900"] + files
    if k:
        cmd += ["-k", k]
    env = _env(lib)
    if order:        # thread interleaving of the emulator (by index / reverse / random): a kernel that cares has a data race
        env["EMU_ORDER"] = order
    if par:          # the blocks of a grid on `par` OS threads at the same time: races BETWEEN blocks (atomics, claims, look-back)
        env["EMU_PAR"] = str(par)
    return subprocess.Popen(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)


DUMPS = {}      # --dump-outputs directories of the two bench jobs


@pytest.fixture(scope="module")
def jobs(tmp_path_factory):
    sys.path.insert(0, EMU)
    import build_emu
    lib = build_emu.build()
    t = lambda f: os.path.join("tests", f)  # noqa: E731
    procs = {
        # round-2 kernels that have not run on a GPU yet — memoised chunk encode (k_encode2.cuh), bpe_replay / resume, the
        # special-token front end (k_special.cuh), file / shard entry points — and bpe_decode
        "new_kernels": _pytest(lib, [t("test_gpu_zy_encode2.py"), t("test_gpu_zz_resume.py"), t("test_gpu_zz_file.py"), t("test_gpu_zz_special.py"), t("test_gpu_zz_gpt2.py"), t("test_gpu_zz_gpt4.py"), t("test_gpu_zz_hist.py"), t("test_gpu_zz_golden_r2.py"),
                                       t("test_gpu_decode.py")], order="random", par=3),
        # kernels already validated on B200s, as a check of the emulator itself (golden vectors of the reference)
        "validated_kernels": _pytest(lib, [t("test_gpu_parity.py")],
                                     "wikipedia or taylorswift or small_cases or primitives or long_runs or table_growth or rescan"),
        "splitter": _pytest(lib, [t("test_gpu_split.py")], "not piecewise", order="reverse"),
        # the sharded loop on 2..4 emulated GPUs (threads): NCCL-style collectives and the NVLink peer-memory kernels
        "sharded": subprocess.Popen([sys.executable, os.path.join(EMU, "emu_sharded.py"), "2:collective", "2:p2p", "3:p2p", "4:p2p"],
                                    cwd=ROOT, env=_env(lib), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True),
    }
    procs["filter"] = _pytest(lib, [t("test_gpu_zz_filter.py")], order="random", par=3)
    # __graft_entry__.smoke(), the call the driver makes on cuda:0 before the bench
    procs["smoke"] = subprocess.Popen([sys.executable, "-c", "import __graft_entry__ as g; g.smoke()"], cwd=ROOT, env=_env(lib),
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    procs["fuzz"] = subprocess.Popen([sys.executable, os.path.join(EMU, "emu_fuzz_encode.py"), "120", "7"], cwd=ROOT, env=dict(_env(lib), EMU_PAR="3"),
                                     stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    # special-token front end (device) against the unmodified reference class (its answers: tests/golden/golden_fuzz_special.json)
    procs["fuzz_special"] = subprocess.Popen([sys.executable, os.path.join(EMU, "emu_fuzz_special.py")], cwd=ROOT, env=_env(lib),
                                             stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    # train() / encode() / save() of the classes against the unmodified reference classes on random small texts
    # (their answers: tests/golden/golden_fuzz_train.json)
    procs["fuzz_train"] = subprocess.Popen([sys.executable, os.path.join(EMU, "emu_fuzz_train_ref.py")], cwd=ROOT, env=_env(lib),
                                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    bench_args = ["--size-mib", "1", "--steps", "6", "--warmup", "3", "--strong-mib", "2", "--strong-sparse-at", "24", "--strong-check", "16",
                  "--encode-gb", "0.002", "--encode-merges", "200", "--encode-train-mib", "1", "--leg-budget-s", "600"]
    benv = dict(_env(lib), BPE_BENCH_EMU="1")
    dump = tmp_path_factory.mktemp("bench_outputs")
    DUMPS.update(bench1=str(dump / "one"), bench2=str(dump / "two"))
    procs["bench1"] = subprocess.Popen([sys.executable, "bench.py", "--full-merges", "40", "--dump-outputs", DUMPS["bench1"]] + bench_args, cwd=ROOT, env=benv,
                                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    procs["bench2"] = subprocess.Popen([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                                        "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), "bench.py", "--gpus", "2",
                                        "--dump-outputs", DUMPS["bench2"]] + bench_args,
                                       cwd=ROOT, env=benv, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    yield procs
    for p in procs.values():
        if p.poll() is None:
            p.kill()


def _finish(jobs, name, timeout=1500):
    p = jobs[name]
    try:
        out, _ = p.communicate(timeout=timeout)
    except subprocess.TimeoutExpired:
        p.kill()
        out, _ = p.communicate()
        pytest.fail(f"emulator job {name} did not finish in {timeout} s\n{out[-3000:]}")
    assert p.returncode == 0, f"emulator job {name} failed\n{out[-6000:]}"
    return out


def test_emu_new_kernels_encode2_resume_decode(jobs):
    out = _finish(jobs, "new_kernels")
    assert " passed" in out and "failed" not in out


def test_emu_validated_kernels_against_reference_goldens(jobs):
    out = _finish(jobs, "validated_kernels")
    assert " passed" in out and "failed" not in out


def test_emu_gpt4_splitter(jobs):
    out = _finish(jobs, "splitter")
    assert " passed" in out and "failed" not in out


def test_emu_sharded_loop_collective_and_p2p(jobs):
    out = _finish(jobs, "sharded")
    assert "emu sharded ok" in out
    assert out.count("bit-exact on every rank") == 12


def test_emu_segment_filter_training(jobs):
    out = _finish(jobs, "filter")
    assert " passed" in out and "failed" not in out


def test_emu_smoke_entry_point(jobs):
    assert "smoke ok" in _finish(jobs, "smoke")


def test_emu_encode_fuzz_under_guard_pages(jobs):
    assert "emu fuzz encode ok" in _finish(jobs, "fuzz")


def test_emu_special_tokens_fuzz_against_the_reference_class(jobs):
    assert "emu fuzz special ok" in _finish(jobs, "fuzz_special")


def test_emu_train_fuzz_against_the_reference_classes(jobs):
    assert "emu fuzz train ok" in _finish(jobs, "fuzz_train")


def _bench_line(jobs, name):
    p = jobs[name]
    try:
        out, err = p.communicate(timeout=1500)
    except subprocess.TimeoutExpired:
        p.kill()
        out, err = p.communicate()
        pytest.fail(f"{name} did not finish\n{err[-3000:]}")
    assert p.returncode == 0, err[-6000:]
    lines = [ln for ln in out.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, out[-2000:]          # the contract: ONE JSON line
    d = json.loads(lines[0])
    # --dump-outputs: the merges and counts of the K timed steps, float64
    m, c = (np.load(os.path.join(DUMPS[name], f + ".npy")) for f in ("merges", "counts"))
    assert m.dtype == c.dtype == np.float64 and m.shape == (d["steps"], 2) and c.shape == (d["steps"],)
    assert m[:4].astype(int).tolist() == d["first_pairs"] and (c > 0).all()
    return d


CONTRACT_KEYS = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                 "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline")


def test_emu_bench_one_rank_every_leg(jobs):
    d = _bench_line(jobs, "bench1")
    for k in CONTRACT_KEYS:
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 6 and d["gpu_launches"] > 0 and "workload" in d["config"]
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["cpu_baseline"]["kind"] == "port"
    assert d["full_run"]["parity_all_merges"] is True and d["full_run"]["merges"] == 40
    assert d["cfg2"]["basic_equals_reference_golden"] is True and d["cfg2"]["regex_equals_reference_golden"] is True
    assert d["strong_cfg4"]["parity_vs_oracle"]["equal"] is True
    assert d["encode_cfg5"]["parity"]["equal"] is True and d["encode_cfg5"]["memo"]["fallback_pieces"] == 0
    assert d["hist_packed"]["same_merges"] is True and d["e2e"]["hist_kernel"] == "k_hist_dense"
    assert d["full_run_filtered"]["same_merges_as_full_run"] is True and d["full_run_filtered"]["merges"] == 40
    test_emu_bench_one_rank_every_leg.sha = d["strong_cfg4"]["merges_sha16"]


def test_emu_bench_two_ranks_every_leg(jobs):
    d = _bench_line(jobs, "bench2")
    for k in CONTRACT_KEYS:
        assert k in d, k
    assert d["n_gpus"] == 2 and d["config"]["consistent"] is True and d["config"]["exchange_used"] == "collective"
    assert d["strong_cfg4"]["parity_vs_oracle"]["equal"] is True
    assert d["encode_cfg5"]["parity"]["equal"] is True
    sha1 = getattr(test_emu_bench_one_rank_every_leg, "sha", None)
    if sha1 is not None:      # strong scaling: the same corpus on 1 and on 2 ranks gives the same merges
        assert d["strong_cfg4"]["merges_sha16"] == sha1


def test_emulator_is_not_a_product_path():
    """Nothing under minbpe_b200/ may reach the emulator build or its header."""
    for dirpath, _, files in os.walk(os.path.join(ROOT, "minbpe_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".inl", ".h", ".c")):
                text = open(os.path.join(dirpath, f), encoding="utf-8", errors="replace").read()
                assert "libb200bpe_emu" not in text and '#include "cuda_emu.h"' not in text and "emu/_build" not in text, f
