"""CPU tests (no GPU): the C-ABI library loads and exports every symbol include/gort_b200.h declares,
fails loudly without a GPU (no CPU fallback), and its host-side LUT text formatter reproduces the
reference's "-W" bytes.  No compute calls are made here."""
import ctypes as C
import json
import os
import re
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

import gort_b200

ROOT = Path(__file__).resolve().parent.parent
GOLD = ROOT / "tests" / "golden"


def header_functions():
    text = (ROOT / "include" / "gort_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(gort_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = gort_b200.load_library()
    names = header_functions()
    assert len(names) >= 20
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing
    # and the Python binding knows about all of them
    assert sorted(gort_b200.ABI_SYMBOLS) == names


def test_no_torch_types_in_the_abi():
    text = (ROOT / "include" / "gort_b200.h").read_text()
    assert "torch" not in text.lower() and "at::" not in text and "std::" not in text


def test_library_is_sm100a_native():
    # the toolkit that built the library (gort_b200/csrc/Makefile) when cuobjdump is not on PATH
    tool = shutil.which("cuobjdump") or str(Path(os.environ.get("CUDA_HOME", "/usr/local/cuda")) / "bin" / "cuobjdump")
    if not Path(tool).exists():
        pytest.skip("cuobjdump unavailable")
    out = subprocess.run([tool, "-lelf", str(ROOT / "gort_b200" / "libgort_b200.so")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert "sm_100a" in out.stdout


def test_create_fails_loudly_without_gpu():
    lib = gort_b200.load_library()
    if lib.gort_device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(gort_b200.GortError) as ei:
        gort_b200.Gort(0)
    assert "no CPU path" in str(ei.value)


def test_lut_text_layout_matches_reference_bytes(tmp_path):
    """gort_lut_write_text on the reference's LUT doubles must give the reference's "-W" bytes
    (gortt.c:124-126), and reading them back must restore rows 0..89 and the k_open pair."""
    gold = np.load(GOLD / "ref_vectors.npz")
    cases = {c["name"]: c for c in json.loads((GOLD / "cli_cases.json").read_text())}
    lut = gold["lut_full"][0]                      # structure 0 is "-LAI 4.0"
    p = tmp_path / "w.txt"
    n = gort_b200.lut_write_text(lut, str(p))
    text = p.read_text()
    assert n == len(text)
    assert text == cases["write_lut"]["stdout"]
    assert text == (GOLD / "lut_lai4.txt").read_text()
    back = gort_b200.lut_read_text(str(p))
    keep = np.r_[0:90, 91:181, 182, 183]
    # %0.40f is exact for values >= ~1e-24 and truncates below that (SURVEY.md 8c)
    big = np.abs(lut[keep]) > 1e-20
    assert np.array_equal(back[keep][big], lut[keep][big])
    assert np.all(np.abs(back[keep][~big] - lut[keep][~big]) < 1e-39)
    assert back[90] == 0.0 and back[181] == 0.0


def test_q08_lut_text(tmp_path):
    gold = np.load(GOLD / "ref_vectors.npz")
    cases = {c["name"]: c for c in json.loads((GOLD / "cli_cases.json").read_text())}
    p = tmp_path / "w.txt"
    gort_b200.lut_write_text(gold["lut_q08"][0], str(p))
    assert p.read_text() == cases["write_lut_q08"]["stdout"]


def test_structure_from_options_matches_reference_cli_derivation():
    # float-typed -LAI: 3.7 is 3.7000000476837158 (SURVEY.md App. B5)
    st = gort_b200.structure_from_options(hb=2, br=1.5, pcc=0.6, lai=3.7)
    r, b = 10.0, 15.0
    lam = float(np.float32(0.6)) / (r * r * np.pi)
    assert st[1] == r and st[2] == b and st[3] == 30.0 and st[4] == 60.0 and st[0] == lam
    assert st[5] == float(np.float32(3.7)) * 3.0 / (lam * r * r * np.pi * b * 4.0)


CLI = ROOT / "gort_b200" / "bin" / "gortt"


@pytest.mark.parametrize("name", ["err_unknown_option", "err_unknown_argument"])
def test_cli_argument_errors_match_reference(name):
    """Option errors are raised before the GPU is touched, so they can be checked on a CPU box."""
    if not CLI.exists():
        pytest.skip("gortt CLI not built")
    case = {c["name"]: c for c in json.loads((GOLD / "cli_cases.json").read_text())}[name]
    r = subprocess.run(["gortt"] + case["args"], executable=str(CLI), input=case["stdin"], capture_output=True, text=True)
    assert (r.returncode, r.stdout, r.stderr) == (case["rc"], case["stdout"], case["stderr"])


def test_cli_usage_exits_zero():
    if not CLI.exists():
        pytest.skip("gortt CLI not built")
    r = subprocess.run([str(CLI), "-u"], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout == "" and "usage:" in r.stderr and "-q08_pn_kopen" in r.stderr
