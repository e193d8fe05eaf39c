"""GPU tier: the exact kernel composition of the BASELINE headline (single level of 4096-frame partitions: fused
block kernel k_fir_level0 in its cluster form + per-block k_fir_mac + time-batched k_fir_mac_batch on three streams)
against the COMPILED reference (oracle/_ref, fir_p.c unmodified) on random data long enough for every partition to meet
non-zero blocks, at batch depth 4/6/8 -- and the same for the opt-in one-kernel-per-block pipeline (k_fir_pipe,
DSP_B200_FIR_PIPE=1): more channels than SMs (a CTA walks two or three channels), shared filter, selectors, ragged
calls mixed in, 2048-frame partitions; BASELINE config 3 (64 channels) at full size."""
import os
from contextlib import contextmanager

import numpy as np
import pytest

from conftest import rms

pytestmark = pytest.mark.gpu
RMS_TOL = 1e-10
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def ref_sample(name):
    """Rows of the compiled reference's output on a test's own input (tests/golden/make_golden.py)."""
    return np.load(os.path.join(GOLDEN, name + ".npz"))


@contextmanager
def env(**kw):
    """Plan-time switches of the library are read with getenv() when the operator is planned."""
    old = {k: os.environ.get(k) for k in kw}
    for k, v in kw.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = str(v)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def write_ir(tmp_path, h):
    p = os.path.join(str(tmp_path), "ir_%d_%d.f64" % h.shape)
    np.ascontiguousarray(h, dtype="<f8").tofile(p)
    return p


# <path>_t<near depth>[_f<far depth>][_u|_s]: _u = every tier for all channels every T-th block, _s = one residue class
# of channels per block (_u2: the far tier in two turns, half the channels each), _m = the per-block MAC and the batch class as one grid; defaults at 32 partitions: no far tier,
# staggered, two launches
VARIANTS = ["pipe_t4", "legacy_t4", "legacy_t4_m", "legacy_t4_f0_u", "legacy_t4_f8_s", "legacy_t4_f8_u", "legacy_t4_f8_u2", "legacy_t4_f12_u", "legacy_t4_f12_s", "legacy_t6_f12_s",
            "legacy_t6_f0_u", "legacy_t8_f0_u", "legacy_t8_f0_s"]


@pytest.mark.parametrize("variant", VARIANTS)
def test_headline_composition_against_compiled_reference(gpu_lib, have_ref, tmp_path, variant):
    """8 contiguous channels (a multiple of 4: the cluster form of the pre-pipeline kernel is taken too), per-channel
    131072-tap IRs, 48 random blocks of 4096 frames: partitions up to p = 31 all meet non-zero blocks, 10+ batched
    V spectra of the near tier and 3 windows of the far tier are consumed.  Reference = fir_p.c compiled unmodified
    (its own 32/256/4096 partition plan)."""
    from oracle import restate
    fs, C, taps, F, nblk = 48000, 8, 131072, 4096, 48
    h = np.stack([restate.bench_ir(taps, c) for c in range(C)], axis=1)
    rng = np.random.default_rng(2024)
    x = rng.standard_normal((nblk * F, C)) * 0.2
    if have_ref:
        from oracle import ref
        r = ref.RefChain("fir_p -t pcm -e double -c %d -r %d %s" % (C, fs, write_ir(tmp_path, h)), fs, C)
        want = np.concatenate([r.run(x[i:i + F]) for i in range(0, nblk * F, F)])
        r.close()
    else:
        want = restate.fir_stream(x, h)
    parts = variant.split("_")
    pipe, t = parts[0], parts[1][1:]
    far = next((q[1:] for q in parts[2:] if q[0] == "f"), None)
    stag = "0" if ("u" in parts[2:] or "u2" in parts[2:]) else "1" if "s" in parts[2:] else None
    with env(DSP_B200_FIR_PIPE="1" if pipe == "pipe" else "0", DSP_B200_FIR_T=t, DSP_B200_FIR_T2=far, DSP_B200_FIR_STAGGER=stag,
             DSP_B200_FIR_MERGE="1" if "m" in parts[2:] else None, DSP_B200_FIR_FAR_CLASSES="2" if "u2" in parts[2:] else None):
        ch = gpu_lib.Chain(fs, C).add_fir(h, block_hint=F)
        plan = ch.describe()[0]
    assert plan["levels"] == [{"B": 4096, "P": 32}] and plan["t_batch"] == int(t), plan
    assert plan["pipe"] == (1 if pipe == "pipe" else 0), plan
    if pipe == "pipe":
        assert plan["pipe_pf"] == int(t) + 2 and plan["t_far"] == 0, plan
    else:
        assert plan["t_far"] == (0 if far is None else int(far)), plan
        assert plan["stagger"] == (int(stag) if stag is not None else (1 if plan["t_far"] == 0 else 0)), plan
        assert plan["merge"] == (1 if "m" in parts[2:] else 0), plan
        if plan["t_far"] and not plan["stagger"]:
            # whole launches of the far tier for all channels, or on request for halves of them in turns
            assert plan["far_classes"] == (2 if "u2" in parts[2:] else 1), plan
    got = np.concatenate([ch.run(x[i:i + F]).copy() for i in range(0, nblk * F, F)])
    ch.close()
    assert got.shape == want.shape
    assert rms(got - want) <= RMS_TOL, (variant, rms(got - want))
    assert np.max(np.abs(got - want)) <= 1e-9
    g = ref_sample("ref_headline")
    assert got.shape[0] == g["frames"]
    assert rms(got[g["rows"]] - g["y"]) <= RMS_TOL, (variant, rms(got[g["rows"]] - g["y"]))
    assert np.max(np.abs(got[g["rows"]] - g["y"])) <= 1e-9


@pytest.mark.parametrize("pipe", [1, 0])
@pytest.mark.parametrize("taps,shared", [(30000, True), (50000, True), (50000, False), (9000, False)])
def test_pipe_more_channels_than_sms(gpu_lib, taps, shared, pipe):
    """300 channels: the persistent grid has one CTA per SM, so most CTAs walk two channels (ring, sbuf hand-over and
    barrier phases cross a channel boundary).  30000 taps = 8 partitions (all summed in the kernel, no batch), 50000 =
    13 (batched tail), 9000 = 3.  8 distinct signals tiled over the channels; the first 8 channels against the
    oracle, the rest bit-identical to them (shared IR) or against their own IRs (per-channel, checked on a sample)."""
    from oracle import restate
    fs, C, F, nblk = 48000, 300, 4096, 17
    rng = np.random.default_rng(taps)
    base = rng.standard_normal((nblk * F, 8)) * 0.2
    reps = (C + 7) // 8
    x = np.tile(base, (1, reps))[:, :C]
    if shared:
        h = restate.bench_ir(taps)
    else:
        h = np.stack([restate.bench_ir(taps, c % 5) for c in range(C)], axis=1)
    with env(DSP_B200_FIR_PIPE=pipe):
        ch = gpu_lib.Chain(fs, C).add_fir(h, block_hint=F)
        plan = ch.describe()[0]
    assert plan["pipe"] == pipe and len(plan["levels"]) == 1, plan
    got = np.concatenate([ch.run(x[i:i + F]).copy() for i in range(0, nblk * F, F)])
    ch.close()
    if shared:
        want = restate.fir_stream(base, h)
        assert rms(got[:, :8] - want) <= RMS_TOL, rms(got[:, :8] - want)
        assert np.array_equal(got, np.tile(got[:, :8], (1, reps))[:, :C])
    else:
        for c in (0, 1, 7, 147, 148, 149, 155, 299):
            want = restate.fir_stream(x[:, c:c + 1], h[:, c:c + 1])
            assert rms(got[:, c:c + 1] - want) <= RMS_TOL, (c, rms(got[:, c:c + 1] - want))
        # channels with the same signal and the same IR must agree bit for bit whichever CTA / iteration computed them
        assert np.array_equal(got[:, 0], got[:, 40]) and np.array_equal(got[:, 3], got[:, 203])


@pytest.mark.parametrize("pipe,taps,far", [(1, 60000, None), (0, 60000, None), (0, 120000, 12), (0, 120000, 8), (0, 120000, 0)])
def test_pipe_selector_latency_and_ragged_mix(gpu_lib, pipe, taps, far):
    """The block kernel behind a scattered selector, writing into the compact buffer of fir's latency ring, with
    whole blocks and ragged calls alternating on the same state (general path <-> fused / pipeline kernel, batched V kept
    current by both).  120000 taps = 30 partitions: both tiers of the batched tail."""
    from oracle import restate
    fs, C, F = 48000, 10, 4096
    rng = np.random.default_rng(77)
    sel = [c in (0, 2, 3, 4, 7, 9) for c in range(C)]
    h = np.stack([restate.bench_ir(taps, c) for c in range(sum(sel))], axis=1)
    for lat in (0, 8192):
        N = 22 * F + 333
        x = rng.standard_normal((N, C)) * 0.2
        want = restate.fir_stream(x, h, selector=sel, latency=lat)
        with env(DSP_B200_FIR_PIPE=pipe, DSP_B200_FIR_T2=far, DSP_B200_FIR_STAGGER="1" if far == 12 else None):
            ch = gpu_lib.Chain(fs, C).add_fir(h, selector=sel, latency=lat, block_hint=F)
            plan = ch.describe()[0]
        assert plan["pipe"] == pipe and plan["t_batch"] == 4 and plan["t_far"] == (far or 0), plan
        cuts = [0, F, 2 * F, 2 * F + 100, 3 * F, 4 * F, 5 * F, 6 * F, 7 * F, 7 * F + 1, 8 * F - 1, 8 * F, 9 * F, 10 * F, 11 * F, 12 * F,
                12 * F + 2000, 14 * F, 15 * F, 16 * F, 17 * F, 18 * F, 19 * F, 20 * F, 21 * F, 22 * F, N]
        got = np.concatenate([ch.run(x[a:b]).copy() for a, b in zip(cuts[:-1], cuts[1:])])
        assert rms(got - want) <= RMS_TOL, (lat, rms(got - want))
        for c in range(C):
            if not sel[c]:
                assert np.array_equal(got[:, c], x[:, c])
        # reset, then the same stream in whole blocks only
        ch.reset()
        got2 = np.concatenate([ch.run(x[i:i + F]).copy() for i in range(0, N, F)])
        assert rms(got2 - want) <= RMS_TOL, (lat, rms(got2 - want))
        ch.close()


@pytest.mark.parametrize("taps,pipe,far", [(20000, 1, None), (70000, 1, None), (20000, 0, None), (70000, 0, None), (70000, 0, 12), (140000, 0, 16),
                                           (140000, 0, None)])
def test_2048_frame_partitions(gpu_lib, taps, pipe, far):
    """Blocks of 2048 frames (the CLI default): a single level of 2048-frame partitions -- 10, 35 and 69 of them --
    through the fused kernel's two-CTA cluster form + MAC + one or two batch tiers (far tier of 8 from 48 partitions
    on, 12 and 16 on request), and through the 2048-point instantiation of the pipeline kernel.  8 channels: two clusters."""
    from oracle import restate
    fs, C, F = 48000, 8, 2048
    rng = np.random.default_rng(taps)
    h = np.stack([restate.bench_ir(taps, c) for c in range(C)], axis=1)
    N = (40 if taps < 100000 else 90) * F
    x = rng.standard_normal((N, C)) * 0.2
    want = restate.fir_stream(x, h)
    with env(DSP_B200_FIR_PIPE=pipe, DSP_B200_FIR_T2=far):
        ch = gpu_lib.Chain(fs, C).add_fir(h, block_hint=F)
        plan = ch.describe()[0]
    assert plan["pipe"] == pipe and plan["levels"][0]["B"] == 2048 and len(plan["levels"]) == 1, plan
    if not pipe:
        P = plan["levels"][0]["P"]
        want_far = far if far else (8 if P >= 48 else 0)
        assert plan["t_far"] == (want_far if P >= 2 * want_far + 2 + 4 else 0), plan
        assert plan["stagger"] == (1 if P - 6 >= 16 and plan["t_far"] == 0 else 0), plan
    got = np.concatenate([ch.run(x[i:i + F]).copy() for i in range(0, N, F)])
    ch.close()
    assert rms(got - want) <= RMS_TOL, rms(got - want)


def test_2048_frame_blocks_two_levels_on_request(gpu_lib):
    """DSP_B200_FIR_SINGLE_MIN=4096 brings back the 2048 + 4096 plan (upper level on the side stream, its tail
    time-batched there)."""
    from oracle import restate
    fs, C, F, taps = 48000, 4, 2048, 70000
    rng = np.random.default_rng(5)
    h = np.stack([restate.bench_ir(taps, c) for c in range(C)], axis=1)
    x = rng.standard_normal((40 * F, C)) * 0.2
    want = restate.fir_stream(x, h)
    with env(DSP_B200_FIR_SINGLE_MIN="4096"):
        ch = gpu_lib.Chain(fs, C).add_fir(h, block_hint=F)
        plan = ch.describe()[0]
    assert [L["B"] for L in plan["levels"]] == [2048, 4096] and plan["tail_pf"] == 1 and plan["t_batch"] == 4, plan
    got = np.concatenate([ch.run(x[i:i + F]).copy() for i in range(0, 40 * F, F)])
    ch.close()
    assert rms(got - want) <= RMS_TOL, rms(got - want)


def test_config3_64_channels_full_size(gpu_lib, have_ref, tmp_path):
    """BASELINE config 3 at its own shape: fir_p, 131072-tap per-channel IRs, 64 channels, 4096-frame blocks, 40
    blocks of the reference's sweep + per-channel tones; channels 0..3 against the compiled reference, a further sample of
    channels against the oracle's plain convolution."""
    from oracle import restate
    fs, C, taps, F, nblk = 48000, 64, 131072, 4096, 40
    h = np.stack([restate.bench_ir(taps, c) for c in range(C)], axis=1)
    x = restate.sgen_sine(fs, C, nblk * F, 20.0, 20000.0) * 0.5
    t = np.arange(nblk * F)[:, None] / fs
    x += 0.25 * np.sin(2 * np.pi * (100.0 + np.arange(C)[None, :]) * t)
    ch = gpu_lib.Chain(fs, C).add_fir(h, block_hint=F)
    got = np.concatenate([ch.run(x[i:i + F]).copy() for i in range(0, nblk * F, F)])
    ch.close()
    if have_ref:
        from oracle import ref
        r = ref.RefChain("fir_p -t pcm -e double -c 4 -r %d %s" % (fs, write_ir(tmp_path, h[:, :4])), fs, 4)
        want = np.concatenate([r.run(x[i:i + F, :4]) for i in range(0, nblk * F, F)])
        r.close()
        assert rms(got[:, :4] - want) <= RMS_TOL, rms(got[:, :4] - want)
    g = ref_sample("ref_config3")
    assert got.shape[0] == g["frames"]
    assert rms(got[g["rows"], :4] - g["y"]) <= RMS_TOL, rms(got[g["rows"], :4] - g["y"])
    for c in (5, 31, 32, 63):
        want = restate.fir_stream(x[:, c:c + 1], h[:, c:c + 1])
        assert rms(got[:, c:c + 1] - want) <= RMS_TOL, (c, rms(got[:, c:c + 1] - want))


def test_fir_selector_leaves_a_slab_empty(gpu_lib):
    """A channel-selective shared-IR filter on a chain cut into slabs: the slab that holds no selected channel is a
    pure pass-through and must not try to plan (it kept no taps)."""
    from oracle import restate
    fs, C, F = 48000, 8, 1024
    h = restate.bench_ir(3000)
    sel = [c == 1 for c in range(C)]
    rng = np.random.default_rng(1)
    x = rng.standard_normal((5 * F, C)) * 0.2
    want = restate.fir_stream(x, h, selector=sel)
    ch = gpu_lib.Chain(fs, C, slabs_per_device=4).add_fir(h, selector=sel)
    got = np.concatenate([ch.run(x[i:i + F]).copy() for i in range(0, 5 * F, F)])
    ch.close()
    assert rms(got - want) <= RMS_TOL
    for c in range(C):
        if not sel[c]:
            assert np.array_equal(got[:, c], x[:, c])
