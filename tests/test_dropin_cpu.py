"""CPU tier of the drop-in boundary: the relinked chain runtime loads, CPU effects still work through
it, and a GPU effect fails its init() loudly (returns NULL -> chain build fails) without a device."""
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
DROPIN = os.path.join(HERE, "dropin", "_build", "libdsp_dropin.so")


def test_dropin_library_without_gpu():
    if not os.path.exists(DROPIN):
        pytest.skip("drop-in harness not built (needs /root/reference at build time)")
    import dsp_b200
    from oracle import ref
    c = ref.RefChain("remix 1 0", 48000, 2, lib_path=DROPIN)      # reference remix.c, still CPU: swaps the channels
    x = np.stack([np.ones(16), np.zeros(16)], axis=1)
    y = c.run(x)
    assert np.array_equal(y[:, 0], x[:, 1]) and np.array_equal(y[:, 1], x[:, 0])
    c.close()
    if dsp_b200.device_count() < 1:
        with pytest.raises(ValueError):
            ref.RefChain("eq 1k 1.0 3", 48000, 2, lib_path=DROPIN)
        # "!" lets an effect fail without aborting the chain build (effects_chain.c:455-458)
        c = ref.RefChain("remix 1 0 ! eq 1k 1.0 3", 48000, 2, lib_path=DROPIN)
        assert c.effect_names() == ["remix"]


def test_shim_exports_reference_symbols():
    """The replacement objects export exactly the symbols the reference's biquad.o fir.o fir_p.o hilbert.o
    resample.o export (SURVEY.md 8b)."""
    import subprocess
    objdir = os.path.join(os.path.dirname(HERE), "oracle", "_ref", "dropin", "shim")
    if not os.path.isdir(objdir):
        pytest.skip("shim objects not built")
    want = {"biquad.o": {"biquad_effect_init", "biquad_init", "biquad_reset", "biquad_init_using_type"},
            "gain.o": {"gain_effect_init"},
            "fir.o": {"fir_effect_init", "fir_effect_init_with_filter"},
            "fir_p.o": {"fir_p_effect_init", "fir_p_effect_init_with_filter"},
            "hilbert.o": {"hilbert_effect_init"}, "resample.o": {"resample_effect_init"}}
    for obj, syms in want.items():
        out = subprocess.run(["nm", "-g", "--defined-only", os.path.join(objdir, obj)], stdout=subprocess.PIPE, text=True).stdout
        have = {line.split()[-1] for line in out.splitlines() if " T " in line}
        assert syms <= have, (obj, syms - have)


def test_align_entry_point_and_fallback_symbols():
    """shim/align.c takes over align_effect_insert (align.h:27); the reference's align.o stays linked under
    ref_align_effect_insert (renamed with objcopy) as the host implementation for chains without GPU effects."""
    import subprocess
    root = os.path.dirname(HERE)
    obj, ref = os.path.join(root, "oracle", "_ref", "dropin", "shim", "align.o"), os.path.join(root, "oracle", "_ref", "dropin", "ref", "align.o")
    if not (os.path.exists(obj) and os.path.exists(ref)):
        pytest.skip("shim objects not built")
    nm = lambda p: {l.split()[-1] for l in subprocess.run(["nm", "-g", "--defined-only", p], stdout=subprocess.PIPE, text=True).stdout.splitlines() if " T " in l}
    assert "align_effect_insert" in nm(obj)
    assert nm(ref) == {"ref_align_effect_insert"}


def test_cpu_chains_keep_the_reference_align(have_ref):
    """A chain without GPU effects that needs alignment (delay.c hands its whole-sample part to the align pass,
    delay.c:153-157,199) gets the reference's own align effect through the fallback -- same output as the pure
    reference, no device needed."""
    if not os.path.exists(DROPIN) or not have_ref:
        pytest.skip("drop-in harness / compiled reference not built")
    from oracle import ref
    chain = ":0 delay 37S : remix 0 1"
    x = np.random.default_rng(0).standard_normal((500, 2))
    a = ref.RefChain(chain, 48000, 2)
    b = ref.RefChain(chain, 48000, 2, lib_path=DROPIN)
    assert a.effect_names() == b.effect_names()
    ya, ca = a.process(x, 128)
    yb, cb = b.process(x, 128)
    assert ca == cb and np.array_equal(ya, yb)


def test_frontend_library_and_ladspa_plugin_load():
    """The drop-in as a library (shim/frontend.c) and as the reference's LADSPA plugin (ladspa_dsp.c unmodified):
    both load and expose their entry points; without a device a GPU effect makes the chain build fail (no fallback)."""
    import ctypes as C
    import dsp_b200
    from dsp_b200 import frontend
    if not frontend.available():
        pytest.skip("frontend library not built (needs /root/reference at build time)")
    L = frontend.lib()
    for n in ("dspfront_chain_new", "dspfront_chain_run", "dspfront_chain_time", "dspfront_chain_free"):
        assert hasattr(L, n)
    c = frontend.DropinChain("remix 1 0", 48000, 2)       # reference effect through the library frontend
    y = c.run(np.stack([np.ones(8), np.zeros(8)], axis=1))
    assert np.array_equal(y[:, 1], np.ones(8))
    c.close()
    if dsp_b200.device_count() < 1:
        with pytest.raises(ValueError):
            frontend.DropinChain("eq 1k 1.0 3", 48000, 2)
    plugin = os.path.join(HERE, "dropin", "_build", "ladspa_dsp_b200.so")
    if os.path.exists(plugin):
        os.environ.setdefault("LADSPA_DSP_CONFIG_PATH", "/nonexistent")
        P = C.CDLL(plugin)
        assert hasattr(P, "ladspa_descriptor")
