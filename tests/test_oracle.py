"""CPU tier: the oracle itself.  (1) the FFTW3 shim behind the compiled reference against numpy;
(2) the compiled reference against the committed golden vectors (regeneration check);
(3) the numpy restatement (oracle/restate.py) against the golden vectors, i.e. against the
reference's own arithmetic.  Nothing here touches the product."""
import ctypes as C
import glob
import os

import numpy as np
import pytest

from conftest import rms

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    return {k: z[k] for k in z.files}


def test_golden_fixtures_present():
    names = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*.npz")))
    assert {"gain", "biquad", "fir_p", "fir_p_2ch", "fir", "fir_direct", "hilbert", "resample_up", "resample_down",
            "resample_2x", "chain"} <= set(names)


def test_fftw_shim_against_numpy():
    """oracle/fftw3_shim.c, the FFT backend of the compiled reference, built on its own by oracle/Makefile."""
    L = C.CDLL(os.path.join(os.path.dirname(GOLDEN), "..", "oracle", "_ref", "libfftw3_shim.so"))
    L.fftw_plan_dft_r2c_1d.restype = C.c_void_p
    L.fftw_plan_dft_r2c_1d.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_uint]
    L.fftw_plan_dft_c2r_1d.restype = C.c_void_p
    L.fftw_plan_dft_c2r_1d.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_uint]
    L.fftw_execute_dft_r2c.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.fftw_execute_dft_c2r.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.fftw_destroy_plan.argtypes = [C.c_void_p]
    rng = np.random.default_rng(0)
    for n in [1, 2, 3, 4, 5, 7, 9, 16, 18, 49, 64, 100, 121, 1176, 1280, 2352, 8192, 2 * 3 * 5 * 7 * 11 * 13, 194, 101]:
        x = rng.standard_normal(n)
        X = np.zeros(n // 2 + 1, dtype=np.complex128)
        p = L.fftw_plan_dft_r2c_1d(n, None, None, 0)
        L.fftw_execute_dft_r2c(p, x.ctypes.data, X.ctypes.data)
        want = np.fft.rfft(x)
        assert np.max(np.abs(X - want)) <= 1e-13 * max(1.0, np.max(np.abs(want))), n
        q = L.fftw_plan_dft_c2r_1d(n, None, None, 0)
        y = np.zeros(n)
        inp = want.copy()
        L.fftw_execute_dft_c2r(q, inp.ctypes.data, y.ctypes.data)
        assert np.max(np.abs(y / n - x)) <= 1e-12, n
        L.fftw_destroy_plan(p)
        L.fftw_destroy_plan(q)


@pytest.mark.parametrize("name", ["gain", "biquad", "fir_p", "fir_p_2ch", "fir", "fir_direct", "hilbert",
                                  "resample_up", "resample_down", "resample_2x", "chain"])
def test_compiled_reference_reproduces_golden(have_ref, name):
    if not have_ref:
        pytest.skip("compiled reference not available")
    from oracle import ref
    g = load(name)
    c = ref.RefChain(str(g["chain"]), int(g["fs"]), int(g["channels"]), dir=GOLDEN)
    y, counts = c.process(g["x"], int(g["block"]))
    assert list(counts) == list(g["counts"])
    assert np.array_equal(y, g["y"])


def test_restated_sgen_matches_reference():
    """Against the compiled reference's sgen output for the same specs (golden/ref_sgen.npz, make_golden.py)."""
    from oracle import restate
    g = load("ref_sgen")
    a = g["tone"]                           # sgen "sine+4800S", 48 kHz, 2 channels
    b = restate.sgen_sine(48000, 2, 4800)
    assert a.shape == b.shape and np.max(np.abs(a - b)) < 1e-12
    a = g["sweep"]                          # sgen "sine:freq=20-20k+4800S", 48 kHz, 1 channel
    b = restate.sgen_sine(48000, 1, 4800, 20.0, 20000.0)
    assert a.shape == b.shape and np.max(np.abs(a - b)) < 1e-9


def test_restated_biquad_against_golden():
    from oracle import restate
    g = load("biquad")
    # the golden chain: eq 31.25 1.4 -2 | eq 1k 1.0 3 | :0,2 lowshelf 200 0.7 4 | : highpass 20 0.7 | allpass_1 500
    import dsp_b200
    fs = int(g["fs"])
    ident = np.array([1.0, 0, 0, 0, 0])
    stages = [
        [dsp_b200.biquad_design(13, fs, 31.25, 1.4, -2.0)] * 4,
        [dsp_b200.biquad_design(13, fs, 1000.0, 1.0, 3.0)] * 4,
        [dsp_b200.biquad_design(14, fs, 200.0, 0.7, 4.0) if k in (0, 2) else ident for k in range(4)],
        [dsp_b200.biquad_design(8, fs, 20.0, 0.7)] * 4,
        [dsp_b200.biquad_design(3, fs, 500.0)] * 4,
    ]
    y = restate.biquad_cascade(g["x"], np.array(stages))
    assert np.max(np.abs(y - g["y"])) < 1e-12


@pytest.mark.parametrize("name,ir,sel,fc", [("fir_p", "ir700.f64", [1, 0, 1], 1), ("fir_p_2ch", "ir300x2.f64", [1, 0, 1], 2),
                                            ("fir", "ir700.f64", None, 1)])
def test_restated_fir_against_golden(name, ir, sel, fc):
    from oracle import restate
    g = load(name)
    taps = np.fromfile(os.path.join(GOLDEN, ir), dtype="<f8").reshape(-1, fc)
    x = g["x"]
    n_out = g["y"].shape[0]
    xz = np.concatenate([x, np.zeros((n_out - x.shape[0], x.shape[1]))])
    y = restate.fir_stream(xz, taps, selector=sel, out_frames=n_out)
    assert np.max(np.abs(y - g["y"])) < 1e-13


def test_restated_hilbert_against_golden():
    from oracle import restate
    g = load("hilbert")
    x = g["x"]
    n_out = g["y"].shape[0]
    xz = np.concatenate([x, np.zeros((n_out - x.shape[0], x.shape[1]))])
    y = restate.fir_stream(xz, restate.hilbert_taps(255), out_frames=n_out)
    assert np.max(np.abs(y - g["y"])) < 1e-13


@pytest.mark.parametrize("name,fs_out", [("resample_up", 48000), ("resample_down", 32000), ("resample_2x", 88200)])
def test_restated_resample_against_golden(name, fs_out):
    from oracle import restate
    g = load(name)
    r = restate.Resampler(int(g["fs"]), fs_out, int(g["channels"]))
    y, counts = r.process(g["x"], int(g["block"]))
    assert list(counts) == list(g["counts"])
    assert rms(y - g["y"]) < 1e-13
