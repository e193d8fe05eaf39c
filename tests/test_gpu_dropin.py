"""GPU tier, drop-in level (SURVEY.md T4): the reference's OWN chain runtime -- effects_chain.c (parser,
optimizer/merge, align insertion, drain bookkeeping), effect.c, align.c, util.c, fir_util.c, sgen.c, all
unmodified -- linked against the shim's replacement objects (shim/*.c -> libdspb200.so), driven through
the same driver as the pure reference (oracle/ref_driver.c).  Same chain strings, same blocks: outputs
must agree to the tolerance and per-call frame counts must be identical.  Also runs the relinked CLI."""
import os
import subprocess

import numpy as np
import pytest

from conftest import rms

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden")
DROPIN = os.path.join(HERE, "dropin", "_build", "libdsp_dropin.so")
CLI_GPU = os.path.join(ROOT, "shim", "_build", "dsp_b200")
CLI_REF = os.path.join(ROOT, "oracle", "_ref", "dsp_ref")
RMS_TOL = 1e-10

NAMES = ["gain", "biquad", "fir_p", "fir_p_2ch", "fir", "fir_direct", "hilbert", "resample_up", "resample_down",
         "resample_2x", "chain",
         # -a / -c alignment: fir_get_offset -> ref -> channel_offsets -> the reference's align pass (effects_chain.c:744-864)
         "fir_p_align", "fir_align_end", "hilbert_c", "hilbert_pc",
         # biquad -r: the reference's reverse-IIR design, run as a device FIR (shim/riir.c)
         "riir"]
LADSPA = os.path.join(HERE, "dropin", "_build", "ladspa_dsp_b200.so")


def load(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    return {k: z[k] for k in z.files}


@pytest.fixture(scope="module")
def dropin(gpu_lib):
    if not os.path.exists(DROPIN):
        pytest.fail("tests/dropin/_build/libdsp_dropin.so missing (linked by __graft_entry__.build() from the objects oracle/Makefile builds where the reference's sources are present)")
    from oracle import ref
    return ref


@pytest.mark.parametrize("name", NAMES)
def test_dropin_golden(dropin, name):
    g = load(name)
    c = dropin.RefChain(str(g["chain"]), int(g["fs"]), int(g["channels"]), dir=GOLDEN, lib_path=DROPIN)
    y, counts = c.process(g["x"], int(g["block"]))
    assert c.fs_out == int(g["out_fs"])
    assert list(counts) == list(g["counts"])
    assert y.shape == g["y"].shape
    assert rms(y - g["y"]) <= RMS_TOL, rms(y - g["y"])
    c.close()


def test_dropin_alignment_effects_are_the_references(dropin):
    """With -a / -c the GPU effect reports (latency, -ref) through channel_offsets and the reference's own alignment
    pass appends its `align` effect: same effect list as the pure reference recorded in the golden file."""
    for name in ("fir_p_align", "fir_align_end", "hilbert_c", "hilbert_pc"):
        g = load(name)
        c = dropin.RefChain(str(g["chain"]), int(g["fs"]), int(g["channels"]), dir=GOLDEN, lib_path=DROPIN)
        names, want = c.effect_names(), [str(e) for e in g["effects"]]
        c.close()
        # the GPU effects may have merged with their neighbours (hilbert + eq -> one device chain); what must agree is
        # the alignment: one `align`, at the end, as in the reference
        assert names.count("align") == want.count("align") == 1 and names[-1] == want[-1] == "align", (name, names, want)
        assert names[0] == want[0], (name, names, want)


def test_dropin_merge_fuses_gpu_effects(dropin):
    """effects_chain_optimize() (effects_chain.c:605-641) + the shim's merge hook: runs of GPU effects become one."""
    c = dropin.RefChain("eq 100 1.0 2 eq 1k 1.0 -2 lowshelf 200 0.7 3 fir_p coefs:0.5,0.25,0.125,0.0625,0.03,0.01,0.005,"
                        "0.002,0.001,0.0005,0.0002,0.0001,0.00005,0.00002,0.00001,0.000005,0.000002,0.000001,0.0000005,"
                        "0.0000002,0.0000001,0.00000005,0.00000002,0.00000001,0.000000005,0.000000002,0.000000001,0.0000000005,"
                        "0.0000000002,0.0000000001,0.00000000005,0.00000000002,0.00000000001 eq 5k 2.0 1", 48000, 2, lib_path=DROPIN)
    assert len(c.effect_names()) == 1, c.effect_names()
    c.close()
    # `add` is not reorderable but adjacent merging keeps the signal order: still one device chain, same result
    spec = "eq 100 1.0 2 eq 1k 1.0 -2 add 0.001 eq 5k 2.0 1"
    c = dropin.RefChain(spec, 48000, 2, lib_path=DROPIN)
    assert len(c.effect_names()) == 1, c.effect_names()
    x = np.random.default_rng(0).standard_normal((3000, 2)) * 0.1
    y, _ = c.process(x, 700)
    c.close()
    if dropin.available():
        r = dropin.RefChain(spec, 48000, 2)
        want, _ = r.process(x, 700)
        assert rms(y - want) <= RMS_TOL
    # a reference CPU effect that is not reorderable splits the run: two GPU groups around it
    c = dropin.RefChain("eq 100 1.0 2 eq 1k 1.0 -2 noise -100 eq 5k 2.0 1", 48000, 2, lib_path=DROPIN)
    assert c.effect_names() == ["eq", "noise", "eq"], c.effect_names()
    c.close()
    # a reorderable CPU effect (delay.c) is hopped over, as the reference's own optimizer does for its effects
    c = dropin.RefChain("eq 100 1.0 2 delay 5S eq 5k 2.0 1", 48000, 2, lib_path=DROPIN)
    assert c.effect_names()[:2] == ["eq", "delay"] and "eq" not in c.effect_names()[1:], c.effect_names()
    c.close()


def test_dropin_matches_reference_on_c2(dropin, have_ref):
    """Config 2 shape: gain + 10 eq, 16 channels, 4096-frame blocks, reference sgen sweep."""
    if not have_ref:
        pytest.skip("compiled reference did not travel")
    chain = "gain -12 " + " ".join("eq %s 1.4 %s" % (f, g) for f, g in zip(
        ["31.25", "62.5", "125", "250", "500", "1k", "2k", "4k", "8k", "16k"], ["-2", "1.5", "-1", "2", "-1.5", "1", "-2", "1.5", "-1", "2"]))
    x = dropin.sgen("sine:freq=20-20k+20000S", 48000, 16, 20000)
    a = dropin.RefChain(chain, 48000, 16)
    b = dropin.RefChain(chain, 48000, 16, lib_path=DROPIN)
    assert b.effect_names() == ["gain"]                # gain + ten biquads: ONE device chain (one H2D/D2H per block)
    ya, ca = a.process(x, 4096)
    yb, cb = b.process(x, 4096)
    assert ca == cb
    assert rms(ya - yb) <= RMS_TOL, rms(ya - yb)


def test_dropin_cli(dropin, tmp_path, have_ref):
    """The relinked CLI (unmodified dsp.c) against the reference CLI, raw float64 out, bit layout identical."""
    if not (os.path.exists(CLI_GPU) and os.path.exists(CLI_REF)):
        pytest.skip("CLI builds did not travel")
    args = ["-q", "-b", "1024", "-t", "sgen", "-c", "4", "-r", "44100", "sine:freq=50-15k+30000S", "-o", "-t", "pcm", "-e", "double"]
    chain = ["gain", "-6", "eq", "200", "1.0", "3", ":0,1", "hilbert", "-p", "255", ":", "fir_p", "-t", "pcm", "-e", "double",
             "-c", "1", "-r", "44100", os.path.join(GOLDEN, "ir700.f64"), "resample", "48k"]
    outs = []
    for exe, name in ((CLI_REF, "ref.f64"), (CLI_GPU, "gpu.f64")):
        out = str(tmp_path / name)
        r = subprocess.run([exe] + args + [out] + chain, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
        outs.append(np.fromfile(out, dtype="<f8").reshape(-1, 4))
    assert outs[0].shape == outs[1].shape and outs[0].shape[0] > 30000
    assert rms(outs[0] - outs[1]) <= RMS_TOL, rms(outs[0] - outs[1])


def test_watch_reloads_gpu_chain_on_its_worker_thread(dropin, tmp_path):
    """The reference's `watch` effect (watch.c:60-123) rebuilds the watched chain on ITS worker thread -- GPU effect
    init (device allocations, filter transforms, the library's process-global tables) and, after the crossfade,
    destroy -- while the caller's thread is inside run() of the old chain; during the crossfade both chains run on the
    same input.  Before the first reload the output must equal the plain chain exactly; through three reloads
    (init on the worker thread, crossfade of two GPU chains, destroy of the old one) every block must come back
    whole and finite."""
    import threading
    import time
    fs, C, F = 48000, 4, 1024
    ir = os.path.join(GOLDEN, "ir700.f64")
    chain_a = "eq 1k 1.0 3 fir_p -t pcm -e double -c 1 -r 48000 %s" % ir
    chain_b = "fir_p -t pcm -e double -c 1 -r 48000 %s eq 300 0.7 -2 hilbert -p 127" % ir
    path = str(tmp_path / "watched.txt")
    with open(path, "w") as f:
        f.write(chain_a + "\n")
    w = dropin.RefChain("watch %s" % path, fs, C, lib_path=DROPIN)
    plain = dropin.RefChain(chain_a, fs, C, lib_path=DROPIN)
    rng = np.random.default_rng(3)
    x0 = rng.standard_normal((F, C)) * 0.2
    assert np.array_equal(w.run(x0), plain.run(x0))
    plain.close()
    stop = threading.Event()

    def rewriter():
        for i in range(3):
            time.sleep(0.7)
            with open(path, "w") as f:
                f.write((chain_b if i % 2 == 0 else chain_a) + "\n")
        stop.set()
    t = threading.Thread(target=rewriter)
    t.start()
    n = 0
    t_end = None
    while True:
        y = w.run(rng.standard_normal((F, C)) * 0.2)
        assert y.shape == (F, C) and np.all(np.isfinite(y)) and np.max(np.abs(y)) < 10.0
        n += 1
        if stop.is_set() and t_end is None:
            t_end = time.time() + 1.8        # one more poll interval + the crossfade
        if t_end is not None and time.time() > t_end:
            break
    t.join()
    assert n > 100
    w.close()


def test_c_abi_is_thread_safe_across_chains(gpu_lib):
    """One thread keeps calling run_host() on a chain while another builds, plans, runs and destroys other chains
    (different FFT sizes: the twiddle tables and the profiling map are process-global).  The first thread's output
    must be bit-identical to a single-threaded run."""
    import threading
    from oracle import restate
    fs, C, F = 48000, 6, 2048
    rng = np.random.default_rng(8)
    h = np.stack([restate.bench_ir(9000, c) for c in range(C)], axis=1)
    xs = [rng.standard_normal((F, C)) * 0.2 for _ in range(60)]
    ref_chain = gpu_lib.Chain(fs, C).add_fir(h, block_hint=F)
    want = [ref_chain.run(x).copy() for x in xs]
    ref_chain.close()
    errors = []
    done = threading.Event()

    def churn():
        k = 0
        try:
            while not done.is_set():
                taps = [300, 1500, 5000, 20000][k % 4]
                blk = [64, 256, 1024, 4096][(k // 2) % 4]
                c = gpu_lib.Chain(fs, 3).add_biquad(np.array([gpu_lib.biquad_design(13, fs, 500.0, 1.0, 2.0)])).add_fir(restate.bench_ir(taps), block_hint=blk)
                c.run(np.ones((blk, 3)) * 0.1)
                c.run(np.ones((blk + 7, 3)) * 0.1)
                c.close()
                k += 1
        except Exception as e:          # pragma: no cover
            errors.append(e)
    t = threading.Thread(target=churn)
    t.start()
    ch = gpu_lib.Chain(fs, C).add_fir(h, block_hint=F)
    got = [ch.run(x).copy() for x in xs]
    done.set()
    t.join()
    ch.close()
    assert not errors, errors
    for a, b in zip(want, got):
        assert np.array_equal(a, b)


def test_ladspa_frontend_runs_gpu_chain(dropin, have_ref, tmp_path):
    """The reference's LADSPA frontend (ladspa_dsp.c, unmodified, -DLADSPA_FRONTEND -DSYMMETRIC_IO) linked against the
    shim objects: load the plugin as a LADSPA host would (ladspa_descriptor -> instantiate -> connect_port -> run),
    float32 ports, against the pure reference chain fed the same float32 samples."""
    import ctypes as C
    if not os.path.exists(LADSPA):
        pytest.fail("tests/dropin/_build/ladspa_dsp_b200.so missing")
    # the LADSPA build has no raw-PCM codec (codec.c:76,121 under LADSPA_FRONTEND): the filter comes as a coefs: literal
    from oracle import restate
    taps = ",".join("%.17g" % v for v in restate.bench_ir(300))
    chain = "gain -3 eq 200 1.0 3 :0 hilbert -p 255 : fir_p coefs:%s" % taps
    cfg = tmp_path / "ladspa_cfg"
    cfg.mkdir()
    (cfg / "config").write_text("input_channels=2\noutput_channels=2\n[effects_chain]\n" + chain + "\n")
    os.environ["LADSPA_DSP_CONFIG_PATH"] = str(cfg)

    class Desc(C.Structure):
        pass
    HANDLE = C.c_void_p
    Desc._fields_ = [("UniqueID", C.c_ulong), ("Label", C.c_char_p), ("Properties", C.c_int), ("Name", C.c_char_p), ("Maker", C.c_char_p),
                     ("Copyright", C.c_char_p), ("PortCount", C.c_ulong), ("PortDescriptors", C.POINTER(C.c_int)), ("PortNames", C.POINTER(C.c_char_p)),
                     ("PortRangeHints", C.c_void_p), ("ImplementationData", C.c_void_p),
                     ("instantiate", C.CFUNCTYPE(HANDLE, C.POINTER(Desc), C.c_ulong)),
                     ("connect_port", C.CFUNCTYPE(None, HANDLE, C.c_ulong, C.POINTER(C.c_float))),
                     ("activate", C.c_void_p), ("run", C.CFUNCTYPE(None, HANDLE, C.c_ulong)), ("run_adding", C.c_void_p),
                     ("set_run_adding_gain", C.c_void_p), ("deactivate", C.c_void_p), ("cleanup", C.CFUNCTYPE(None, HANDLE))]
    L = C.CDLL(LADSPA)          # the constructor reads the config directory
    L.ladspa_descriptor.restype = C.POINTER(Desc)
    L.ladspa_descriptor.argtypes = [C.c_ulong]
    d = L.ladspa_descriptor(0)
    assert d and d.contents.PortCount == 4 and d.contents.Label == b"ladspa_dsp"
    inst = d.contents.instantiate(d, 48000)
    assert inst
    n, nblk = 1000, 6
    rng = np.random.default_rng(12)
    x = (rng.standard_normal((n * nblk, 2)) * 0.2).astype(np.float32)
    ports = [np.zeros(n, dtype=np.float32) for _ in range(4)]
    for i, p in enumerate(ports):
        d.contents.connect_port(inst, i, p.ctypes.data_as(C.POINTER(C.c_float)))
    outs = []
    for b in range(nblk):
        ports[0][:] = x[b * n:(b + 1) * n, 0]
        ports[1][:] = x[b * n:(b + 1) * n, 1]
        d.contents.run(inst, n)
        outs.append(np.stack([ports[2].copy(), ports[3].copy()], axis=1))
    d.contents.cleanup(inst)
    got = np.concatenate(outs).astype(np.float64)
    if have_ref:
        r = dropin.RefChain(chain, 48000, 2)
        want = np.concatenate([r.run(x[b * n:(b + 1) * n].astype(np.float64)) for b in range(nblk)])
        r.close()
        assert got.shape == want.shape
        assert rms(got - want.astype(np.float32).astype(np.float64)) <= 1e-7      # float32 ports


def test_device_chain_continues_across_align_and_resample(dropin, gpu_lib, have_ref):
    """SURVEY.md 8f-1: runs of GPU effects the optimizer cannot merge -- a latency-bearing `fir`, the chain's `align`
    (now a device operator), `biquad -r`, `resample` -- are still one device chain per block: ONE host->device and ONE
    device->host copy per run_effects_chain() call (copy counter of the library), output equal to the reference's."""
    ir = os.path.join(GOLDEN, "ir700.f64")
    cases = [
        # (chain, fs, channels, block): config 5 in miniature; fir's FFT path (latency 700 -> align discards 700 frames)
        # between two biquads and a resampler; reverse IIR + alignment of the other channel + resample
        ("eq 100 1.0 2 eq 1k 1.0 -2 eq 5k 2.0 1 fir_p -t pcm -e double -c 1 -r 44100 %s resample 48k" % ir, 44100, 2, 512),
        ("eq 200 1.0 3 fir -t pcm -e double -c 1 -r 44100 %s eq 3k 1.0 -3 resample 48k" % ir, 44100, 2, 500),
        (":0 highpass -r 2k bw2 : eq 300 1.0 2 resample 44100", 48000, 2, 700),
    ]
    rng = np.random.default_rng(21)
    for chain, fs, C, block in cases:
        x = rng.standard_normal((9 * block, C)) * 0.2
        g = dropin.RefChain(chain, fs, C, lib_path=DROPIN)
        names = g.effect_names()
        outs, counts = [], []
        for i in range(0, x.shape[0], block):
            h0, d0 = gpu_lib.copy_counts()
            y = g.run(x[i:i + block])
            h1, d1 = gpu_lib.copy_counts()
            # (a call that yields no frames yet -- the resampler still filling its first block -- has nothing to copy back)
            assert (h1 - h0, d1 - d0) == (1, 1 if y.shape[0] > 0 else 0), (chain, names, h1 - h0, d1 - d0)
            outs.append(y)
            counts.append(y.shape[0])
        for y in g.drain(block):
            outs.append(y)
            counts.append(y.shape[0])
        g.close()
        got = np.concatenate(outs)
        if have_ref:
            r = dropin.RefChain(chain, fs, C)
            want, wcounts = r.process(x, block)
            r.close()
            assert counts == list(wcounts), (chain, counts[:6], list(wcounts)[:6])
            assert got.shape == want.shape
            assert rms(got - want) <= RMS_TOL, (chain, rms(got - want))
    # and with the hand-off disabled the same chains still agree (every effect on its own device chain)
    os.environ["DSP_B200_NO_LINK"] = "1"
    try:
        chain, fs, C, block = cases[1]
        x = rng.standard_normal((6 * block, C)) * 0.2
        g = dropin.RefChain(chain, fs, C, lib_path=DROPIN)
        got, counts = g.process(x, block)
        g.close()
        if have_ref:
            r = dropin.RefChain(chain, fs, C)
            want, wcounts = r.process(x, block)
            r.close()
            assert counts == list(wcounts) and rms(got - want) <= RMS_TOL
    finally:
        os.environ.pop("DSP_B200_NO_LINK", None)


def test_delay_between_gpu_effects_keeps_one_device_chain(dropin, gpu_lib, have_ref):
    """`delay` hands its whole-sample part to the chain's align pass (delay.c:153-157,199) and is itself reorderable:
    the GPU effects around it still merge into one device chain (one copy in, at most one out per call), the align
    effect the chain appends realises the delays (on the device when it lands next to a GPU effect, else the
    reference's own), and the stream equals the pure reference's."""
    if not have_ref:
        pytest.skip("compiled reference did not travel")
    chain = "eq 1k 1.0 3 :0 delay 37S : eq 200 1.0 2 :1 delay 5S : lowshelf 300 0.7 -2"
    rng = np.random.default_rng(6)
    x = rng.standard_normal((4000, 2)) * 0.2
    a = dropin.RefChain(chain, 48000, 2)
    b = dropin.RefChain(chain, 48000, 2, lib_path=DROPIN)
    assert "align" in b.effect_names()
    ya, ca = a.process(x, 512)
    h0, d0 = gpu_lib.copy_counts()
    yb, cb = b.process(x, 512)
    h1, d1 = gpu_lib.copy_counts()
    assert ca == cb
    assert rms(ya - yb) <= RMS_TOL, rms(ya - yb)
    calls = len(cb)
    assert h1 - h0 == calls and d1 - d0 <= calls, (h1 - h0, d1 - d0, calls)
