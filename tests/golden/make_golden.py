"""Regenerates tests/golden/*.npz from the compiled reference (oracle/_ref, built by oracle/Makefile
where the reference's sources are present):  python tests/golden/make_golden.py [--samples]

Each fixture stores the chain string, stream format, block size, the INPUT (float64) and the
reference's concatenated OUTPUT plus per-call frame counts, so the GPU tests need neither the
reference's sources nor the compiled reference to check parity.  --samples regenerates only the
ref_*.npz files (see reference_samples()).
"""
import os
import shutil
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import ref, restate  # noqa: E402


def save(name, chain, fs, channels, block, x, files=None):
    c = ref.RefChain(chain, fs, channels, dir=HERE)
    y, counts = c.process(x, block)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), chain=chain, fs=fs, channels=channels, block=block,
                        x=x, y=y, counts=np.array(counts), out_fs=c.fs_out, effects=np.array(c.effect_names()))
    print(name, chain, x.shape, "->", y.shape, c.effect_names())


def main():
    rng = np.random.default_rng(20260924)
    # C1: plumbing
    x = ref.sgen("sine+1000S", 48000, 2, 1000)
    save("gain", "gain -6", 48000, 2, 256, x)
    # biquad cascade, selector on one stage
    x = ref.sgen("sine:freq=20-20k+1500S", 48000, 4, 1500) * 0.5
    x[:, 1] *= -0.7
    x[:, 3] = rng.standard_normal(1500) * 0.1
    save("biquad", "eq 31.25 1.4 -2 eq 1k 1.0 3 :0,2 lowshelf 200 0.7 4 : highpass 20 0.7 allpass_1 500", 48000, 4, 300, x)
    # fir_p, mono IR from a coefs: literal would be long; use a raw f64 file next to the fixtures
    h = restate.bench_ir(700)
    h.astype("<f8").tofile(os.path.join(HERE, "ir700.f64"))
    x = ref.sgen("sine:freq=20-20k+2000S", 48000, 3, 2000) * 0.9
    x[:, 2] = rng.standard_normal(2000) * 0.2
    save("fir_p", ":0,2 fir_p -t pcm -e double -c 1 -r 48000 ir700.f64", 48000, 3, 256, x)
    # per-channel IR (2 selected channels -> 2 filter columns)
    h2 = np.stack([restate.bench_ir(300, 1), restate.bench_ir(300, 2)], axis=1)
    h2.astype("<f8").tofile(os.path.join(HERE, "ir300x2.f64"))
    save("fir_p_2ch", ":0,2 fir_p -t pcm -e double -c 2 -r 48000 ir300x2.f64", 48000, 3, 1000, x)
    # fir (FFT path, latency len; the chain appends align) and the <=16-tap direct form
    save("fir", "fir -t pcm -e double -c 1 -r 48000 ir700.f64", 48000, 3, 512, x)
    save("fir_direct", "fir coefs:0.5,0.25,-0.125,0.0625,0.03", 48000, 3, 100, x)
    save("hilbert", "hilbert -p 255", 48000, 3, 333, x)
    # -a alignment (fir_util.c:187-205 -> channel_offsets -> the chain's align pass, effects_chain.c:744-864): the
    # filtered channels ask for a negative delay (peak index / offset from the end / centre tap), the chain turns the
    # difference into `align` effects on the OTHER channels.  Drop-in tier only (the align pass is reference code).
    save("fir_p_align", ":0,2 fir_p -a -t pcm -e double -c 1 -r 48000 ir700.f64", 48000, 3, 256, x)
    save("fir_align_end", ":1 fir -a-100S -t pcm -e double -c 1 -r 48000 ir700.f64", 48000, 3, 512, x)
    save("hilbert_c", ":0 hilbert -c 255", 48000, 3, 333, x)
    save("hilbert_pc", ":0,1 hilbert -p -c 255 :2 eq 1k 1.0 3", 48000, 3, 333, x)
    # reverse IIR (biquad -r, reverse_iir.c): the linear-phase LR4 crossover of examples/crossover_lr4_2kHz_riir_linphase
    # without its remix (4 channels in), two -r sections per band merged by the chain, plus a lone -r section
    x4 = np.concatenate([x, x[:, :1] * 0.5], axis=1)
    save("riir", ":0,1 highpass 2k bw2 highpass -r 2k bw2 : :2,3 lowpass 2k bw2 lowpass -r 2k bw2 : :1 eq -r 500 1.0 4", 48000, 4, 500, x4)
    # resample both ways, ragged blocks, drain included
    x = ref.sgen("sine:freq=1k+3000S", 44100, 2, 3000) * 0.8
    x[:, 1] = rng.standard_normal(3000) * 0.3
    save("resample_up", "resample 48000", 44100, 2, 500, x)
    save("resample_down", "resample 32000", 44100, 2, 777, x)
    save("resample_2x", "resample x2", 44100, 2, 64, x[:1500])
    # full chain (C5 in miniature)
    save("chain", "gain -3 eq 100 1.0 2 eq 5k 2.0 -3 fir_p -t pcm -e double -c 1 -r 44100 ir700.f64 resample 48000", 44100, 2, 512, x)
    reference_samples()


def sample_rows(n, k, seed):
    """A fixed, sorted sample of k of n rows (all of them when n <= k)."""
    return np.arange(n) if n <= k else np.sort(np.random.default_rng(seed).choice(n, k, replace=False))


def run_blocks(chain, fs, x, sizes):
    """The reference chain fed x in calls of the given sizes: (concatenated output, per-call frame counts)."""
    r = ref.RefChain(chain, fs, x.shape[1], dir=HERE)
    outs, pos = [], 0
    for n in sizes:
        outs.append(r.run(x[pos:pos + n]))
        pos += n
    r.close()
    return np.concatenate(outs), np.array([y.shape[0] for y in outs])


def save_sample(name, y, k, seed, counts=None, **extra):
    rows = sample_rows(y.shape[0], k, seed)
    kw = dict(extra, rows=rows, y=y[rows], frames=y.shape[0])
    if counts is not None:
        kw["counts"] = counts
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **kw)
    print(name, y.shape, "->", kw["y"].shape)


def reference_samples():
    """The reference outputs the larger GPU tests and the host-side checks compare against, at the tests' own inputs
    (the inputs are rebuilt here exactly as the tests build them).  Outputs too large to commit are stored as a fixed
    sample of rows; `rows` indexes the test's full output."""
    import tempfile
    tmp = tempfile.mkdtemp()
    # tests/test_abi.py: the coefficient design, every type / width type the test walks
    args = []
    for t in range(1, 16):
        for wt in (1, 2, 3, 4, 5):
            if wt in (2, 3) and t not in (14, 15):
                continue
            for f0, w, g in [(1000, 0.7, 3.0), (31.25, 1.4, -2), (16000, 0.5, 6), (100, 2.0, -9.5)]:
                args.append((t, 48000, f0, w, g, 0, wt))
    args += [(t, 44100, 50, 0.7, 20, 0.5, 1) for t in (16, 17)]
    coefs = np.array([ref.biquad_design(a[0], a[1], a[2], a[3], a[4], a[5], a[6]) for a in args])
    np.savez_compressed(os.path.join(HERE, "ref_biquad_design.npz"), args=np.array(args, dtype=np.float64), coefs=coefs)
    # tests/test_oracle.py: the reference's signal generator (a tone on two channels, a sweep)
    a = ref.sgen("sine+4800S", 48000, 2, 4800)
    b = ref.sgen("sine:freq=20-20k+4800S", 48000, 1, 4800)
    np.savez_compressed(os.path.join(HERE, "ref_sgen.npz"), tone=a, sweep=b)
    # tests/test_gpu_headline.py: fir_p, 8 channels x 131072-tap IRs, 48 blocks of 4096 random frames
    fs, C, taps, F, nblk = 48000, 8, 131072, 4096, 48
    h = np.stack([restate.bench_ir(taps, c) for c in range(C)], axis=1)
    x = np.random.default_rng(2024).standard_normal((nblk * F, C)) * 0.2
    ir = os.path.join(tmp, "ir_headline.f64")
    h.astype("<f8").tofile(ir)
    y, _ = run_blocks("fir_p -t pcm -e double -c %d -r %d %s" % (C, fs, ir), fs, x, [F] * nblk)
    save_sample("ref_headline", y, 512, 1)
    # tests/test_gpu_headline.py: config 3, channels 0..3 of 64, 40 blocks of sweep + per-channel tones
    C, nblk = 64, 40
    h = np.stack([restate.bench_ir(taps, c) for c in range(4)], axis=1)
    x = restate.sgen_sine(fs, C, nblk * F, 20.0, 20000.0) * 0.5
    x += 0.25 * np.sin(2 * np.pi * (100.0 + np.arange(C)[None, :]) * (np.arange(nblk * F)[:, None] / fs))
    ir = os.path.join(tmp, "ir_config3.f64")
    h.astype("<f8").tofile(ir)
    y, _ = run_blocks("fir_p -t pcm -e double -c 4 -r %d %s" % (fs, ir), fs, x[:, :4], [F] * nblk)
    save_sample("ref_config3", y, 512, 2)
    # tests/test_gpu_parity.py: resampling at five rate pairs (1024-frame calls, drained) ...
    rs = {}
    for fi, fo in [(44100, 48000), (48000, 44100), (48000, 96000), (96000, 48000), (44100, 32000)]:
        x = np.random.default_rng(fi + fo).standard_normal((9000, 5)) * 0.3
        x[:, 0] = np.sin(2 * np.pi * 1000.0 * np.arange(9000) / fi)
        y, counts = ref.RefChain("resample %d" % fo, fi, 5).process(x, 1024)
        rows = sample_rows(y.shape[0], 128, fo)
        rs.update({"%d_%d_rows" % (fi, fo): rows, "%d_%d_y" % (fi, fo): y[rows], "%d_%d_counts" % (fi, fo): np.array(counts)})
    np.savez_compressed(os.path.join(HERE, "ref_resample_ratios.npz"), **rs)
    # ... at every channel count of the kernel variants (ragged calls, not drained) ...
    rs = {}
    for C in (1, 2, 4, 6, 36, 132):
        x = np.random.default_rng(C).standard_normal((5000, C)) * 0.3
        y, counts = run_blocks("resample 48000", 44100, x, [1024, 7, 2048, 1, 900, 1020])
        cols = sorted({0, C // 3, C // 2, C - 1})
        rows = sample_rows(y.shape[0], 128, C)
        rs.update({"%d_rows" % C: rows, "%d_cols" % C: np.array(cols), "%d_y" % C: y[rows][:, cols], "%d_counts" % C: counts})
    np.savez_compressed(os.path.join(HERE, "ref_resample_channels.npz"), **rs)
    # ... and config 4's 8 distinct signals, 3 blocks of 4096 frames
    fi, F, nblk = 44100, 4096, 3
    tt = np.arange(nblk * F)[:, None] / fi
    base = np.sin(2 * np.pi * (500.0 + 250.0 * np.arange(8)[None, :]) * tt) * 0.5 + restate.sgen_sine(fi, 8, nblk * F, 20.0, 20000.0) * 0.25
    y, counts = run_blocks("resample 48000", fi, base, [F] * nblk)
    save_sample("ref_config4", y, 256, 4, counts=counts)
    shutil.rmtree(tmp)


if __name__ == "__main__":
    if sys.argv[1:] == ["--samples"]:
        reference_samples()
    else:
        main()
