"""CPU-side checks of the drop-in boundary: the C-ABI library loads, exports every symbol the
header declares, and refuses to work (loudly) without a CUDA device."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, "include", "dsp_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(dspb200_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    import dsp_b200
    L = dsp_b200.lib()
    names = header_functions()
    assert len(names) >= 25
    for n in names:
        assert hasattr(L, n), "libdspb200.so lacks %s" % n
    # and the binding knows a signature for each of them
    from dsp_b200.lib import SIGNATURES
    assert sorted(SIGNATURES) == names


def test_version_and_error_channel():
    import dsp_b200
    assert b"sm_100a" in dsp_b200.lib().dspb200_version()
    assert isinstance(dsp_b200.last_error(), str)


def test_no_cpu_fallback_without_device():
    import dsp_b200
    if dsp_b200.device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(dsp_b200.DspB200Error):
        dsp_b200.Chain(48000, 2)


def test_product_never_imports_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may touch oracle/."""
    pat = re.compile(r"^\s*(from|import)\s+oracle\b|liboracle|libdspref|oracle[./]ref|oracle[./]restate|oracle[./]port", re.M)
    for sub in ("dsp_b200", "shim", "include"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, sub)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".c", ".cpp")):
                    text = open(os.path.join(dirpath, f), errors="replace").read()
                    assert not pat.search(text), "%s reaches into the oracle" % os.path.join(dirpath, f)


def test_host_side_design_matches_reference():
    """biquad.c:111-294 coefficient design, bit for bit (host arithmetic, no GPU needed), against the compiled
    reference's designs of every type and width type (tests/golden/ref_biquad_design.npz, make_golden.py)."""
    import numpy as np
    import dsp_b200
    g = np.load(os.path.join(ROOT, "tests", "golden", "ref_biquad_design.npz"))
    assert len(g["args"]) == 15 * 3 * 4 + 2 * 2 * 4 + 2
    for (t, fs, f0, w, gain, a3, wt), b in zip(g["args"], g["coefs"]):
        a = dsp_b200.biquad_design(int(t), fs, f0, w, gain, a3, int(wt))
        assert np.array_equal(a, b), (t, wt, f0, a, b)


def test_helpers_match_restatement():
    import numpy as np
    import dsp_b200
    from oracle import restate
    assert np.allclose(dsp_b200.hilbert_taps(255), restate.hilbert_taps(255), rtol=0, atol=0)
    for fi, fo in [(44100, 48000), (48000, 44100), (48000, 96000), (96000, 48000), (44100, 32000)]:
        p = dsp_b200.resample_params(fi, fo)
        r = restate.Resampler(fi, fo, 1)
        assert (p["n"], p["d"], p["m"], p["in_len"], p["out_len"], p["out_delay"]) == (r.n, r.d, r.m, r.in_len, r.out_len, r.out_delay)


def test_chain_language_mirror():
    from dsp_b200 import effects
    assert effects.parse_freq("1k") == 1000.0
    assert effects.parse_width("2o") == (2.0, effects.WIDTH_BW_OCT)
    assert effects.parse_width("0.5k") == (500.0, effects.WIDTH_BW_HZ)
    w, t = effects.parse_width("bw4.1")
    assert t == effects.WIDTH_Q and abs(w - 1.0 / (2.0 * __import__("math").sin(3.141592653589793 / 4 * 0.5))) < 1e-15
    assert effects.parse_selector("0,2", 4) == [1, 0, 1, 0]
    assert effects.parse_selector("1-", 4) == [0, 1, 1, 1]
    assert effects.parse_selector("-", 3) == [1, 1, 1]
