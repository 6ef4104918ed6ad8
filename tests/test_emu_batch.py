"""CPU: the batched encode (tests/test_gpu_zz_batch.py) against the kernel SOURCES on the SIMT emulator (tests/emu/), as
tests/test_emu.py does for the other GPU files: once with random thread order inside a block and three blocks of a grid
on OS threads at the same time (races inside and between blocks), once against the UBSan build (alignment of the vector
accesses, shift counts, array bounds)."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "emu")
FILE = os.path.join("tests", "test_gpu_zz_batch.py")


def _run(lib, extra_env):
    env = dict(os.environ)
    env.update(BPE_LIB_PATH=lib, BPE_TEST_SMALL="1", EMU_SMS="2", PYTHONDONTWRITEBYTECODE="1", **extra_env)
    env.pop("PYTEST_CURRENT_TEST", None)
    cmd = [sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", "-p", "no:cacheprovider", FILE]
    return subprocess.Popen(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)


def test_batch_on_the_emulator():
    sys.path.insert(0, EMU)
    import build_emu
    lib = build_emu.build()
    jobs = {"random order, 3 blocks at once": _run(lib, {"EMU_ORDER": "random", "EMU_PAR": "3"})}
    san_env = dict(os.environ, EMU_SANITIZE="1")
    subprocess.check_call([sys.executable, "-c", "import build_emu; build_emu.build(force=True)"], cwd=EMU, env=san_env)
    ubsan = subprocess.run(["g++", "-print-file-name=libubsan.so"], capture_output=True, text=True, check=True).stdout.strip()
    jobs["UBSan build"] = _run(lib.replace(".so", "_ubsan.so"), {"LD_PRELOAD": ubsan})
    for name, p in jobs.items():
        out, _ = p.communicate(timeout=3600)
        assert p.returncode == 0, f"{name}:\n{out[-6000:]}"
        assert " passed" in out and "failed" not in out, f"{name}:\n{out[-3000:]}"
