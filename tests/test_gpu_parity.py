"""GPU tier: seeded inputs at sizes beyond the golden fixtures against the oracle (the compiled
reference when it travelled, else the numpy restatement), plus size-independent properties at
BASELINE.json's full sizes (impulse -> IR, linearity)."""
import os

import numpy as np
import pytest

from conftest import rms

pytestmark = pytest.mark.gpu
RMS_TOL = 1e-10
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def ref_sample(name):
    """Rows of the compiled reference's output on a test's own input (tests/golden/make_golden.py)."""
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def eq_coefs(gpu_lib, fs, n_stages):
    f = [31.25, 62.5, 125, 250, 500, 1000, 2000, 4000, 8000, 16000]
    g = [-2, 1.5, -1, 2, -1.5, 1, -2, 1.5, -1, 2]
    return np.array([gpu_lib.biquad_design(13, fs, f[i], 1.4, g[i]) for i in range(n_stages)])


def test_biquad_c2_cascade(gpu_lib):
    """Config 2 in miniature: 10-stage eq cascade, 64 ch, 4096-frame blocks, sweep + per-channel tones."""
    from oracle import restate
    fs, C, F = 48000, 64, 4096
    coefs = eq_coefs(gpu_lib, fs, 10)
    x = restate.sgen_sine(fs, C, 3 * F, 20.0, 20000.0) * 0.25
    t = np.arange(3 * F)[:, None] / fs
    x += 0.25 * np.sin(2 * np.pi * (100.0 + np.arange(C)[None, :]) * t)
    want = restate.biquad_cascade(x, coefs)
    ch = gpu_lib.Chain(fs, C).add_biquad(coefs)
    got = np.concatenate([ch.run(x[i:i + F]).copy() for i in range(0, 3 * F, F)])
    assert rms(got - want) <= RMS_TOL, rms(got - want)
    # ragged calls, same stream
    ch.reset()
    cuts = [0, 1, 33, 100, 4196, 4197, 9000, 3 * F]
    got2 = np.concatenate([ch.run(x[a:b]).copy() for a, b in zip(cuts[:-1], cuts[1:])])
    assert rms(got2 - want) <= RMS_TOL
    ch.close()


def test_biquad_per_channel_coefficients_and_long_cascade(gpu_lib):
    from oracle import restate
    fs, C, S = 44100, 7, 20      # 20 stages -> two fused operators of <= 16
    rng = np.random.default_rng(3)
    coefs = np.zeros((S, C, 5))
    for s in range(S):
        for c in range(C):
            coefs[s, c] = gpu_lib.biquad_design(13, fs, 40.0 * (1.3 ** s) + 3 * c, 0.7 + 0.1 * c, rng.uniform(-6, 6))
    coefs[3, 2] = [1, 0, 0, 0, 0]
    x = rng.standard_normal((5000, C)) * 0.1
    want = restate.biquad_cascade(x, coefs)
    ch = gpu_lib.Chain(fs, C).add_biquad(coefs)
    assert ch.n_ops == 2
    got = np.concatenate([ch.run(x[i:i + 999]).copy() for i in range(0, 5000, 999)])
    assert rms(got - want) <= RMS_TOL
    ch.close()


@pytest.mark.parametrize("block", [64, 1000, 1024, 2048, 4096])
def test_fir_p_block_sizes(gpu_lib, block):
    from oracle import restate
    fs, C, taps = 48000, 6, 5000
    rng = np.random.default_rng(block)
    h = np.stack([restate.bench_ir(taps, c) for c in range(4)], axis=1)
    sel = [1, 1, 0, 1, 0, 1]
    N = 6 * 4096 + 123
    x = rng.standard_normal((N, C)) * 0.2
    want = restate.fir_stream(x, h, selector=sel)
    ch = gpu_lib.Chain(fs, C).add_fir(h, selector=sel)
    got = np.concatenate([ch.run(x[i:i + block]).copy() for i in range(0, N, block)])
    assert rms(got - want) <= RMS_TOL, rms(got - want)
    assert np.array_equal(got[:, 2], x[:, 2]) and np.array_equal(got[:, 4], x[:, 4])
    ch.close()


def test_fir_p_ragged_calls_and_partition_hint(gpu_lib):
    from oracle import restate
    fs, C, taps = 48000, 3, 3000
    rng = np.random.default_rng(11)
    h = restate.bench_ir(taps)
    N = 20000
    x = rng.standard_normal((N, C)) * 0.2
    want = restate.fir_stream(x, h)
    for hint in (256, 1024):
        ch = gpu_lib.Chain(fs, C).add_fir(h, block_hint=hint)
        cuts = sorted(set([0, N] + list(rng.integers(1, N, 25))))
        got = np.concatenate([ch.run(x[a:b]).copy() for a, b in zip(cuts[:-1], cuts[1:])])
        assert rms(got - want) <= RMS_TOL, (hint, rms(got - want))
        ch.close()


def test_fir_latency_ring(gpu_lib):
    """fir.c's FFT path: same convolution, delayed by len = next_fast_fftw_len(taps)."""
    from oracle import restate
    fs, C, taps = 48000, 2, 700
    rng = np.random.default_rng(5)
    h = restate.bench_ir(taps)
    L = restate.next_fast_fftw_len(taps)
    x = rng.standard_normal((9000, C)) * 0.2
    want = restate.fir_stream(x, h, latency=L)
    for block in (100, 512, 3000):
        ch = gpu_lib.Chain(fs, C).add_fir(h, latency=L)
        got = np.concatenate([ch.run(x[i:i + block]).copy() for i in range(0, 9000, block)])
        assert rms(got - want) <= RMS_TOL, block
        ch.close()


@pytest.mark.parametrize("rates", [(44100, 48000), (48000, 44100), (48000, 96000), (96000, 48000), (44100, 32000)])
def test_resample_ratios(gpu_lib, have_ref, rates):
    from oracle import restate
    fi, fo = rates
    C = 5
    rng = np.random.default_rng(fi + fo)
    x = rng.standard_normal((9000, C)) * 0.3
    x[:, 0] = np.sin(2 * np.pi * 1000.0 * np.arange(9000) / fi)
    if have_ref:
        from oracle import ref
        want, wcounts = ref.RefChain("resample %d" % fo, fi, C).process(x, 1024)
    else:
        want, wcounts = restate.Resampler(fi, fo, C).process(x, 1024)
    ch = gpu_lib.Chain(fi, C).add_resample(fo)
    got, counts = ch.process(x, 1024)
    assert counts == list(wcounts)
    assert rms(got - want) <= RMS_TOL, rms(got - want)
    g, k = ref_sample("ref_resample_ratios"), "%d_%d_" % (fi, fo)
    assert counts == list(g[k + "counts"])
    assert rms(got[g[k + "rows"]] - g[k + "y"]) <= RMS_TOL
    ch.close()


@pytest.mark.parametrize("channels", [1, 2, 4, 6, 36, 132])
def test_resample_channel_counts_pick_every_kernel_variant(gpu_lib, have_ref, channels):
    """channels % 4 == 0 runs on the FP64 tensor cores (k_rs_mma: 4, 36 = a partly filled warp, 132 = a
    partly filled second CTA column), everything else on the FMA kernel (k_rs_poly: pairs for even counts,
    single channels for odd ones); ragged call sizes on top."""
    from oracle import restate
    fi, fo = 44100, 48000
    rng = np.random.default_rng(channels)
    x = rng.standard_normal((5000, channels)) * 0.3
    sizes = [1024, 7, 2048, 1, 900, 1020]
    if have_ref:
        from oracle import ref
        r = ref.RefChain("resample %d" % fo, fi, channels)
    else:
        r = restate.Resampler(fi, fo, channels)
    ch = gpu_lib.Chain(fi, channels).add_resample(fo)
    pos, outs = 0, []
    for n in sizes:
        blk = x[pos:pos + n]
        pos += n
        want = r.run(blk)
        got = ch.run(blk).copy()
        assert got.shape == want.shape
        if want.size:
            assert rms(got - want) <= RMS_TOL
        outs.append(got)
    ch.close()
    g, k = ref_sample("ref_resample_channels"), "%d_" % channels
    assert [y.shape[0] for y in outs] == list(g[k + "counts"])
    assert rms(np.concatenate(outs)[g[k + "rows"]][:, g[k + "cols"]] - g[k + "y"]) <= RMS_TOL


def test_full_size_impulse_response_property(gpu_lib):
    """Headline shape (256 ch x 131072 taps, per-channel IR, 4096-frame blocks): a delta in gives the
    IR back -- a size-independent known answer (SURVEY.md T0)."""
    from oracle import restate
    fs, C, taps, F = 48000, 256, 131072, 4096
    h = np.stack([restate.bench_ir(taps, c) for c in range(C)], axis=1)
    ch = gpu_lib.Chain(fs, C).add_fir(h, block_hint=F)
    x = np.zeros((F, C))
    x[5, :] = 1.0
    x[7, 3] = -0.5
    outs = [ch.run(x).copy()]
    z = np.zeros((F, C))
    for _ in range(taps // F):
        outs.append(ch.run(z).copy())
    y = np.concatenate(outs)
    want = np.zeros_like(y)
    want[5:5 + taps] = h
    want[7:7 + taps, 3] += -0.5 * h[:, 3]
    assert np.max(np.abs(y - want)) <= 1e-13
    ch.close()


def test_full_size_linearity_property(gpu_lib):
    """conv(a x1 + b x2) == a conv(x1) + b conv(x2) on the headline shape with a shared IR."""
    from oracle import restate
    fs, C, taps, F = 48000, 256, 131072, 4096
    h = restate.bench_ir(taps)
    rng = np.random.default_rng(9)
    x1 = rng.standard_normal((3 * F, C)) * 0.2
    x2 = rng.standard_normal((3 * F, C)) * 0.2

    def conv(x):
        ch = gpu_lib.Chain(fs, C).add_fir(h, block_hint=F)
        y = np.concatenate([ch.run(x[i:i + F]).copy() for i in range(0, 3 * F, F)])
        ch.close()
        return y
    y1, y2, y12 = conv(x1), conv(x2), conv(0.5 * x1 - 2.0 * x2)
    assert rms(y12 - (0.5 * y1 - 2.0 * y2)) <= 1e-13
    # and one channel against the oracle's plain convolution
    want = restate.fir_stream(x1[:, 17:18], h)
    assert rms(y1[:, 17:18] - want) <= RMS_TOL


def test_device_resident_mode(gpu_lib):
    """Mode D (run_device on torch-owned buffers and stream) equals mode A."""
    import torch
    from oracle import restate
    fs, C, F = 48000, 16, 1024
    h = restate.bench_ir(3000)
    coefs = eq_coefs(gpu_lib, fs, 4)
    rng = np.random.default_rng(2)
    x = rng.standard_normal((4 * F, C)) * 0.2
    a = gpu_lib.Chain(fs, C).add_biquad(coefs).add_fir(h, block_hint=F)
    b = gpu_lib.Chain(fs, C).add_biquad(coefs).add_fir(h, block_hint=F)
    ya = np.concatenate([a.run(x[i:i + F]).copy() for i in range(0, 4 * F, F)])
    st = torch.cuda.current_stream().cuda_stream
    outs = []
    for i in range(0, 4 * F, F):
        d = torch.from_numpy(x[i:i + F].copy()).cuda()
        n = b.run_device(0, F, d.data_ptr(), d.data_ptr(), st)
        assert n == F
        outs.append(d.cpu().numpy())
    assert np.array_equal(ya, np.concatenate(outs))
    a.close()
    b.close()


def test_submit_wait_equals_synchronous_calls(gpu_lib):
    """dspb200_chain_submit_host/wait with several blocks in flight (rate-changing chain, 3 channel
    slabs, ragged block sizes) gives bit-identical blocks and frame counts to run_host."""
    from oracle import restate
    fs, C = 44100, 12
    h = restate.bench_ir(5000)
    coefs = eq_coefs(gpu_lib, fs, 3)
    rng = np.random.default_rng(5)
    sizes = [1024, 1024, 700, 1024, 1, 2048, 1024, 1024, 333, 1024, 1024, 1024]
    xs = [rng.standard_normal((n, C)) * 0.2 for n in sizes]
    def make():
        return gpu_lib.Chain(fs, C, slabs_per_device=3).add_biquad(coefs).add_fir(h, block_hint=1024).add_resample(48000)
    a, b = make(), make()
    want = [a.run(x).copy() for x in xs]
    ins = [gpu_lib.PinnedArray((2048, C)) for _ in xs]
    outs = [gpu_lib.PinnedArray((b.max_out_frames(2048) + 1, C)) for _ in xs]
    pending, got = [], [None] * len(xs)
    for i, x in enumerate(xs):
        ins[i].array[:len(x)] = x
        n, t = b.submit_raw(len(x), ins[i].ptr, outs[i].ptr)
        pending.append((i, n, t))
        if len(pending) > 4:
            j, m, tj = pending.pop(0)
            b.wait(tj)
            got[j] = outs[j].array[:m].copy()
    for j, m, tj in pending:
        b.wait(tj)
        got[j] = outs[j].array[:m].copy()
    for w, g in zip(want, got):
        assert w.shape == g.shape
        assert np.array_equal(w, g)
    a.close()
    b.close()


def test_in_process_multi_gpu_sharding(gpu_lib):
    """One chain sharded over two GPUs in one process (DSP_B200_DEVICES in the shim): one strided host
    scatter and gather per shard, no collective; bit-identical to the single-GPU chain."""
    if gpu_lib.device_count() < 2:
        pytest.skip("needs 2 GPUs (run under gpurun --gpus 2)")
    from oracle import restate
    fs, C, F = 48000, 12, 1024
    h = np.stack([restate.bench_ir(3000, c) for c in range(C)], axis=1)
    coefs = eq_coefs(gpu_lib, fs, 3)
    rng = np.random.default_rng(4)
    x = rng.standard_normal((5 * F, C)) * 0.2

    def build(devices, slabs):
        return gpu_lib.Chain(fs, C, devices=devices, slabs_per_device=slabs).add_biquad(coefs).add_fir(h, block_hint=F).add_resample(44100)
    a, b = build([0], 1), build([0, 1], 2)
    assert b.n_shards == 4 and {b.shard_info(i)[0] for i in range(4)} == {0, 1}
    ya, ca = a.process(x, F)
    yb, cb = b.process(x, F)
    assert ca == cb
    assert np.array_equal(ya, yb)
    a.close()
    b.close()


@pytest.mark.parametrize("block,taps", [(8192, 70000), (10000, 20000), (65536, 20000), (300, 40000), (40000, 70000), (16384, 30000), (65536, 140000)])
def test_fir_p_large_and_odd_blocks(gpu_lib, block, taps):
    """Partition = 8192 with many partitions (single level, three-kernel path), calls longer than the largest
    partition (bulk form: several whole blocks per launch, with and without a ragged remainder), and a small odd
    block with a long filter (four levels)."""
    from oracle import restate
    fs, C = 48000, 4
    rng = np.random.default_rng(block + taps)
    h = restate.bench_ir(taps)
    N = max(3 * block, 2 * taps) + 77
    x = rng.standard_normal((N, C)) * 0.2
    want = restate.fir_stream(x, h)
    ch = gpu_lib.Chain(fs, C).add_fir(h)
    got = np.concatenate([ch.run(x[i:i + block]).copy() for i in range(0, N, block)])
    plan = ch.describe()[0]
    assert plan["planned"] == 1
    assert rms(got - want) <= RMS_TOL, (plan, rms(got - want))
    ch.close()


@pytest.mark.parametrize("shared", [True, False])
def test_fir_p_bulk_form_mixes_with_ragged_calls(gpu_lib, shared):
    """A plan made for 32768-frame calls (4 blocks of 8192 per launch) fed with calls of every kind: bulk,
    bulk + remainder, tiny, exactly one block, more blocks than the plan holds at once; shared and per-channel IR."""
    from oracle import restate
    fs, C, taps = 48000, 3, 50000
    rng = np.random.default_rng(11)
    h = restate.bench_ir(taps) if shared else np.stack([restate.bench_ir(taps, c) for c in range(C)], axis=1)
    sizes = [32768, 100, 8192, 20000, 32768, 5, 16384 + 8192 - 105, 65536 + 3, 8192, 40000]
    x = rng.standard_normal((sum(sizes), C)) * 0.2
    want = restate.fir_stream(x, h)
    ch = gpu_lib.Chain(fs, C).add_fir(h, block_hint=32768)
    assert ch.describe()[0]["levels"] == [{"B": 8192, "P": 7}]
    outs, pos = [], 0
    for n in sizes:
        outs.append(ch.run(x[pos:pos + n]).copy())
        pos += n
    got = np.concatenate(outs)
    assert rms(got - want) <= RMS_TOL, rms(got - want)
    ch.reset()
    got2 = np.concatenate([ch.run(x[i:i + 32768]).copy() for i in range(0, 3 * 32768, 32768)])
    assert rms(got2 - want[:3 * 32768]) <= RMS_TOL
    ch.close()


@pytest.mark.parametrize("block,taps,shared", [(4096, 60000, True), (4096, 131072, False), (8192, 100000, False), (4096, 13000, True),
                                               (2048, 131072, False), (2048, 40000, True)])
def test_fir_p_single_level_with_tail(gpu_lib, block, taps, shared):
    """Blocks of 2048 frames and up (4096 is the largest partition size of multi-level plans): ONE level,
    its fused kernel sums partitions 0 and 1, the rest arrives as a spectrum accumulated two blocks ahead
    (time-batched when there are enough partitions; 13000 taps = 4 partitions: not batched).  Aligned calls,
    then the same stream in random cuts (general path and fused path interleave on the same state)."""
    from oracle import restate
    fs, C = 48000, 3
    rng = np.random.default_rng(block + taps)
    h = restate.bench_ir(taps) if shared else np.stack([restate.bench_ir(taps, c) for c in range(C)], axis=1)
    N = 14 * block + 1234
    x = rng.standard_normal((N, C)) * 0.2
    want = restate.fir_stream(x, h)
    ch = gpu_lib.Chain(fs, C).add_fir(h, block_hint=block)
    plan = ch.describe()[0]
    assert len(plan["levels"]) == 1 and plan["tail_pf"] == 2, plan
    assert (plan["t_batch"] > 0) == (plan["levels"][0]["P"] >= 11), plan
    got = np.concatenate([ch.run(x[i:i + block]).copy() for i in range(0, N, block)])
    assert rms(got - want) <= RMS_TOL, (plan, rms(got - want))
    ch.reset()
    cuts = sorted(set([0, N, 3 * block, 4 * block, 5 * block, 9 * block] + list(rng.integers(1, N, 12))))
    got2 = np.concatenate([ch.run(x[a:b]).copy() for a, b in zip(cuts[:-1], cuts[1:])])
    assert rms(got2 - want) <= RMS_TOL, (plan, rms(got2 - want))
    ch.close()


@pytest.mark.parametrize("case", ["all8", "window", "scattered", "latency", "biquad_first"])
def test_fir_direct_block_io_variants(gpu_lib, case):
    """Whole aligned blocks on single-level plans are read and written by the fused kernel itself: clusters of four
    adjacent channels when the selected channels are contiguous (all 8; channels 4..11 of 12), one channel per
    CTA otherwise (scattered selector); into the compact buffer of fir's latency ring; and after an in-place
    neighbour in the same chain (in == out)."""
    from oracle import restate
    fs, F, taps = 48000, 4096, 20000
    rng = np.random.default_rng(7)
    C = 8 if case in ("all8", "latency", "biquad_first") else 12
    sel = None
    if case == "window":
        sel = [4 <= c < 12 for c in range(C)]
    if case == "scattered":
        sel = [c in (1, 2, 5, 6, 7, 10, 11, 3) for c in range(C)]
    n_sel = C if sel is None else sum(sel)
    h = np.stack([restate.bench_ir(taps, c) for c in range(n_sel)], axis=1)
    lat = 24576 if case == "latency" else 0
    x = rng.standard_normal((6 * F + 100, C)) * 0.2
    ch = gpu_lib.Chain(fs, C)
    xin = x
    if case == "biquad_first":
        coefs = eq_coefs(gpu_lib, fs, 2)
        ch.add_biquad(coefs)
        xin = restate.biquad_cascade(x, coefs)
    ch.add_fir(h, selector=sel, latency=lat, block_hint=F)
    want = restate.fir_stream(xin, h, selector=sel, latency=lat)
    got = np.concatenate([ch.run(x[i:i + F]).copy() for i in range(0, x.shape[0], F)])
    assert rms(got - want) <= RMS_TOL, (case, rms(got - want))
    ch.close()


def test_full_size_config2_biquad_cascade(gpu_lib):
    """BASELINE config 2 at full size: gain -12 dB + 10 eq stages, 256 channels, 48 kHz, 4096-frame blocks; every
    channel against the restated recurrence (biquad.h:76-92), sweep + per-channel tones as SURVEY 8d prescribes."""
    from oracle import restate
    fs, C, F, nblk = 48000, 256, 4096, 3
    coefs = eq_coefs(gpu_lib, fs, 10)
    x = restate.sgen_sine(fs, C, nblk * F, 20.0, 20000.0) * 0.5
    t = np.arange(nblk * F)[:, None] / fs
    x += 0.25 * np.sin(2 * np.pi * (100.0 + np.arange(C)[None, :]) * t)
    g = 10.0 ** (-12.0 / 20.0)
    want = restate.biquad_cascade(x * g, coefs)
    ch = gpu_lib.Chain(fs, C).add_gain(np.full(C, g)).add_biquad(coefs)
    got = np.concatenate([ch.run(x[i:i + F]).copy() for i in range(0, nblk * F, F)])
    assert rms(got - want) <= RMS_TOL, rms(got - want)
    ch.close()


def test_full_size_config4_resample(gpu_lib, have_ref):
    """BASELINE config 4 at full size: 44100 -> 48000, 1024 channels (tensor-core kernel, 8 CTA columns).  Channels
    c and c + 8 carry the same signal: the first 8 are checked against the oracle, the rest must equal them bit for
    bit (a channel's result may not depend on the lane / warp / CTA that computes it)."""
    from oracle import restate
    fi, fo, C, F, nblk = 44100, 48000, 1024, 4096, 3
    tt = np.arange(nblk * F)[:, None] / fi
    base = np.sin(2 * np.pi * (500.0 + 250.0 * np.arange(8)[None, :]) * tt) * 0.5 + restate.sgen_sine(fi, 8, nblk * F, 20.0, 20000.0) * 0.25
    x = np.tile(base, (1, C // 8))
    if have_ref:
        from oracle import ref
        r = ref.RefChain("resample %d" % fo, fi, 8)
    else:
        r = restate.Resampler(fi, fo, 8)
    ch = gpu_lib.Chain(fi, C).add_resample(fo)
    outs = []
    for i in range(0, nblk * F, F):
        want = r.run(base[i:i + F])
        got = ch.run(x[i:i + F]).copy()
        assert got.shape == (want.shape[0], C)
        assert rms(got[:, :8] - want) <= RMS_TOL
        assert np.array_equal(got, np.tile(got[:, :8], (1, C // 8)))
        outs.append(got[:, :8])
    ch.close()
    g = ref_sample("ref_config4")
    assert [y.shape[0] for y in outs] == list(g["counts"])
    assert rms(np.concatenate(outs)[g["rows"]] - g["y"]) <= RMS_TOL


def test_full_size_config5_chain_share(gpu_lib, have_ref):
    """One GPU's share of BASELINE config 5: 8 eq stages + fir_p 65536 taps (shared IR) + resample 44100 -> 48000,
    256 channels; 4 distinct signals tiled over the channels, checked against the oracle composition."""
    from oracle import restate
    fi, fo, C, F, nblk = 44100, 48000, 256, 4096, 4
    coefs = eq_coefs(gpu_lib, fi, 8)
    h = restate.bench_ir(65536)
    rng = np.random.default_rng(5)
    base = rng.standard_normal((nblk * F, 4)) * 0.2
    x = np.tile(base, (1, C // 4))
    y = restate.fir_stream(restate.biquad_cascade(base, coefs), h)
    r = restate.Resampler(fi, fo, 4)
    ch = gpu_lib.Chain(fi, C).add_biquad(coefs).add_fir(h, block_hint=F).add_resample(fo)
    for i in range(0, nblk * F, F):
        want = r.run(y[i:i + F])
        got = ch.run(x[i:i + F]).copy()
        assert got.shape == (want.shape[0], C)
        assert rms(got[:, :4] - want) <= RMS_TOL
        assert np.array_equal(got, np.tile(got[:, :4], (1, C // 4)))
    ch.close()


def test_align_operator_delays_and_discard(gpu_lib):
    """Device `align` (align.c:35-64): per-channel whole-frame delays through rings that persist across calls of any
    size, the first `discard` frames of the stream dropped (a call returns the tail of its block)."""
    fs, C = 48000, 6
    delays = [0, 3, 700, 1, 0, 5000]
    rng = np.random.default_rng(4)
    N = 12000
    x = rng.standard_normal((N, C))
    for discard in (0, 1300):
        want = np.zeros((N, C))
        for k, d in enumerate(delays):
            want[d:, k] = x[:N - d, k]
        want = want[discard:]
        ch = gpu_lib.Chain(fs, C).add_align(delays, discard)
        cuts = [0, 1, 2, 500, 1299, 1300, 1301, 4000, 4001, 9000, N]
        outs = [ch.run(x[a:b]).copy() for a, b in zip(cuts[:-1], cuts[1:])]
        got = np.concatenate(outs)
        assert got.shape == want.shape, (discard, got.shape, want.shape)
        assert np.array_equal(got, want)
        ch.reset()
        got2 = np.concatenate([ch.run(x[i:i + 4096]).copy() for i in range(0, N, 4096)])
        assert np.array_equal(got2, want)
        ch.close()


def test_fir_replans_after_unrepresentative_first_call(gpu_lib):
    """A first call of 7 frames must not pin 64-frame partitions for the life of the effect: the next, representative
    call (2048 frames) redoes the plan and replays the frames seen so far; the stream is the same as ever."""
    from oracle import restate
    fs, C, taps = 48000, 3, 30000
    rng = np.random.default_rng(17)
    h = np.stack([restate.bench_ir(taps, c) for c in range(C)], axis=1)
    sizes = [7, 2048, 2048, 100, 2048, 2048, 2048, 4096, 2048]
    x = rng.standard_normal((sum(sizes), C)) * 0.2
    want = restate.fir_stream(x, h)
    ch = gpu_lib.Chain(fs, C).add_fir(h)
    outs, pos = [], 0
    for i, n in enumerate(sizes):
        outs.append(ch.run(x[pos:pos + n]).copy())
        pos += n
        if i == 0:
            assert ch.describe()[0]["levels"][0]["B"] == 64
        if i == 1:
            assert ch.describe()[0]["levels"][0]["B"] == 2048, ch.describe()[0]
    got = np.concatenate(outs)
    assert rms(got - want) <= RMS_TOL, rms(got - want)
    ch.close()
