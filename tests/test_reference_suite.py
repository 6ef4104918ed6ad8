"""CPU: the checks of the reference's own test file (karpathy/minbpe tests/test_tokenizer.py) against minbpe_b200 — the
drop-in claim — with the reference's answers stored under tests/golden/ (golden_ref_suite.json), so that every result is
also compared with the unmodified reference.  No GPU here, so the library under the classes is the CPU SIMT emulator build
of the kernel sources (tests/emu/).  The 9 GPT4Tokenizer tests of that file need tiktoken's cl100k_base (a download) and
are not part of it; 12 checks remain."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_test_file_passes_against_minbpe_b200():
    sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
    import build_emu
    lib = build_emu.build()
    env = dict(os.environ, BPE_LIB_PATH=lib, PYTHONDONTWRITEBYTECODE="1")
    env.pop("PYTEST_CURRENT_TEST", None)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "emu", "emu_reference_suite.py")],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "reference suite ok: 12 passed" in r.stdout, r.stdout[-1000:]
