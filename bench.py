#!/usr/bin/env python
"""bench.py -- headline benchmark of the effects-chain hot path on B200.

Metric (BASELINE.json): Msamples/s through a 256-channel x 131072-tap `fir_p` chain, 1 sample =
one double of one channel-frame at the chain input; weak scaling (every GPU owns 256 channels,
independent streams, no collective on the data path).  One "step" = one block of --block frames
(default 4096) x 256 channels through the chain.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [...]                         # the reference's CPU path
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --dump-outputs DIR [...]                       # also write the timed paths' last outputs

Prints ONE JSON line on rank 0.
  value         device-resident throughput (inputs in HBM).  The timed region is closed over EVERY stream the
                chain uses (dspb200_chain_join before the end event), so the look-ahead MAC launches that belong
                to the timed blocks are inside it.
  e2e           the same blocks through the C-ABI host call (dspb200_chain_run_host) from pinned host memory,
                copies inside the timed region.
  roofline      algorithmic HBM bytes of all kernels of a step / step time, against the measured HBM peak, plus a
                per-kernel table (each kernel timed alone).
  cpu_baseline  the compiled reference (oracle/_ref) on this box's host cores over a bounded sample.
  configs       (1 GPU runs) driver-run numbers for BASELINE configs 2-5, the CLI-default 2048-frame block, and
                `e2e_dropin`: run_effects_chain() of the reference's chain runtime with the GPU effects linked in.

With --dump-outputs DIR, rank 0 also writes the block the headline and e2e paths returned in their last timed step
as DIR/<name>.npy (float64, [frames, channels]; at most 64 MB = 64e6 bytes in all, beyond that a fixed, seeded sample
of frames): `device` (the headline's device-resident call), `host` and `host_pipelined` (the two host-call legs of
`e2e`, unless --no-e2e).  The configs are not dumped.  Inputs and IRs are seeded, so two builds run with the same
arguments can be compared output for output.
"""
import argparse
import math
import json
import multiprocessing as mp
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FS = 48000
CHANNELS_PER_GPU = 256
TAPS = 131072
METRIC = "Msamples/s through 256-ch 128k-tap fir_p chain"
UNIT = "Msamples/s"
EQ_F = [31.25, 62.5, 125, 250, 500, 1000, 2000, 4000, 8000, 16000]
EQ_G = [-2, 1.5, -1, 2, -1.5, 1, -2, 1.5, -1, 2]


# ------------------------------------------------------------------------------------------------
# workload definition (SURVEY.md 8d): seeded decaying-noise IR per channel, noise-like input blocks
# ------------------------------------------------------------------------------------------------
def park_miller(seed, count):
    """x -> 48271 x mod (2^31-1) (the reference's pm_rand1_r, util.h:127-148), vectorised."""
    M = np.uint64(0x7fffffff)
    pw = np.array([48271], dtype=np.uint64)
    while pw.shape[0] < count:
        pw = np.concatenate([pw, (pw * pw[-1]) % M])
    return ((pw[:count] * np.uint64(seed)) % M).astype(np.float64)


def make_ir(taps, channel):
    u = 2.0 * park_miller(1 + channel, taps) / 2147483647.0 - 1.0
    h = u * np.exp(-6.9 * np.arange(taps) / taps)
    return h * (0.5 / np.sum(np.abs(h)))


def make_irs(taps, channels, first_channel=0):
    return np.stack([make_ir(taps, first_channel + c) for c in range(channels)], axis=1)


def make_block(frames, channels, seed):
    u = park_miller(1000 + seed, frames * channels) / 2147483647.0 - 0.5
    return u.reshape(frames, channels)


DUMP_LIMIT = 64 * 10 ** 6          # bytes of all files together, .npy headers included
NPY_HEADER_MAX = 4096


def dump_outputs(path, arrays):
    """arrays: name -> [frames, channels].  Each goes to path/<name>.npy as float64; when the files would exceed
    DUMP_LIMIT bytes together, every array is cut to the same fixed, seeded sample of its frames (sorted)."""
    os.makedirs(path, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    budget = DUMP_LIMIT - NPY_HEADER_MAX * len(arrays)
    for name, v in arrays.items():
        if total > budget:
            keep = max(1, v.shape[0] * budget // total)
            v = v[np.sort(np.random.default_rng(0).choice(v.shape[0], keep, replace=False))]
        np.save(os.path.join(path, name + ".npy"), v)


# ------------------------------------------------------------------------------------------------
# host placement: a rank's pinned buffers and its copy-issuing thread belong on its GPU's NUMA node
# ------------------------------------------------------------------------------------------------
def usable_cores():
    """Cores this process may really use: the affinity mask, capped by a cgroup CPU quota if there is one."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(math.ceil(float(q) / float(p)))))
    except Exception:
        pass
    return n


def bind_to_gpu_numa(device):
    """sched_setaffinity to the CPUs of the NUMA node the GPU hangs off (first-touch then places the pinned
    buffers there).  Returns a description for the JSON line, or None when the topology cannot be read."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(device)
        busid = "%04x:%02x:%02x.0" % (bus.pci_domain_id, bus.pci_bus_id, bus.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % busid).read().strip())
        if node < 0:
            return {"pci": busid, "numa_node": node, "bound": False}
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return {"pci": busid, "numa_node": node, "bound": False}
        os.sched_setaffinity(0, cpus)
        return {"pci": busid, "numa_node": node, "bound": True, "cpus": len(cpus)}
    except Exception as e:                                             # topology files missing in this container
        return {"bound": False, "why": str(e)[:80]}


# ------------------------------------------------------------------------------------------------
# clocks during the timed region (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# CPU legs: the compiled reference on host cores (the only place oracle/ is executed here)
# ------------------------------------------------------------------------------------------------
CPU_FLAVOURS = [("O2", "libdspref.so", "-O2"), ("Os", "libdspref_Os.so", "-Os (the reference's own level, GNUmakefile:57)"),
                ("O3", "libdspref_O3.so", "-O3 -march=x86-64-v3 (stand-in for -march=native: built off-box)")]


def _cpu_worker(args):
    lib_path, ir_path, ch, block, warm, steps, seconds = args
    sys.path.insert(0, ROOT)
    from oracle import ref          # checker / baseline only
    c = ref.RefChain("fir_p -t pcm -e double -c %d -r %d %s" % (ch, FS, ir_path), FS, ch, lib_path=lib_path)
    c.run_inplace(block, refill=True)
    for _ in range(warm):
        c.run_inplace(block)
    t0 = time.perf_counter()
    n = 0
    while (steps and n < steps) or (not steps and time.perf_counter() - t0 < seconds):
        c.run_inplace(block)
        n += 1
    dt = time.perf_counter() - t0
    c.close()
    return n, dt


def _cpu_trial(lib_path, ir_path, procs, ch_per_proc, block, warm, steps, seconds):
    ctx = mp.get_context("spawn")
    with ctx.Pool(procs) as pool:
        res = pool.map(_cpu_worker, [(lib_path, ir_path, ch_per_proc, block, warm, steps, seconds)] * procs)
    # every process ran concurrently; job throughput = sum of the per-process rates
    rate = sum(n * block * ch_per_proc / dt for n, dt in res)
    return rate, sum(n for n, _ in res), max(dt for _, dt in res), max(n for n, _ in res)


def cpu_reference_suite(block, sample_s=5.0, runs=3, one_proc_s=3.0, ch_per_proc=2):
    """The reference on the host cores (SURVEY.md 8d): for every build flavour (i) ONE process (fir_p's own <= 3
    worker threads included) and (ii) P processes, each a reference fir_p chain of `ch_per_proc` channels with its own
    131072-tap IRs (channels are independent: this is how the reference would use the box).  P is picked once, from
    2-second trials over {n/4, n/2, n} usable cores; the P-process figure is the median of `runs` samples of
    `sample_s` seconds, with the spread.  fir_p defers most of its arithmetic to worker threads with a two-period
    deadline (fir_p.c:105-114): samples are seconds long so that work is inside them."""
    from oracle import ref
    if not ref.available():
        return None
    ncpu = usable_cores()
    ref_dir = os.path.dirname(ref.LIB_PATH)
    flavours = [(k, os.path.join(ref_dir, f), d) for k, f, d in CPU_FLAVOURS if os.path.exists(os.path.join(ref_dir, f))]
    tmp = tempfile.mkdtemp(prefix="dspb200_bench_")
    ir_path = os.path.join(tmp, "ir.f64")
    make_irs(TAPS, ch_per_proc).astype("<f8").tofile(ir_path)
    out = {"cores_usable": ncpu, "cores_os": os.cpu_count(), "flavours": {}}
    try:
        # process count: 2-second trials over {n/4, n/2, n} usable cores narrow it down, then the two best are measured
        # for a full sample each (fir_p's deferred thread work makes short trials noisy) and the better one is kept
        cands = sorted(set(max(1, ncpu // d) for d in (4, 2, 1)))
        trials = {}
        for p in cands:
            trials[p] = _cpu_trial(flavours[0][1], ir_path, p, ch_per_proc, block, 2, 0, 2.0)[0] / 1e6
        out["process_count_trials_Msps"] = {str(k): round(v, 2) for k, v in trials.items()}
        top = sorted(trials, key=trials.get, reverse=True)[:2]
        finals = {p: _cpu_trial(flavours[0][1], ir_path, p, ch_per_proc, block, 2, 0, sample_s)[0] / 1e6 for p in top}
        out["process_count_finals_Msps"] = {str(k): round(v, 2) for k, v in finals.items()}
        procs = max(finals, key=finals.get)
        for key, path, desc in flavours:
            one = _cpu_trial(path, ir_path, 1, ch_per_proc, block, 2, 0, one_proc_s)[0] / 1e6
            samples = sorted(_cpu_trial(path, ir_path, procs, ch_per_proc, block, 2, 0, sample_s)[0] / 1e6 for _ in range(runs))
            out["flavours"][key] = {"build": desc, "one_process_Msps": one, "n_process_Msps_median": samples[len(samples) // 2],
                                    "n_process_Msps_min": samples[0], "n_process_Msps_max": samples[-1], "processes": procs}
    finally:
        os.remove(ir_path)
        os.rmdir(tmp)
    best = max(out["flavours"], key=lambda k: out["flavours"][k]["n_process_Msps_median"])
    b = out["flavours"][best]
    out.update({"value": b["n_process_Msps_median"], "unit": UNIT, "cores": procs, "kind": "reference", "flavour": best,
                "spread": [b["n_process_Msps_min"], b["n_process_Msps_max"]],
                "sample": "fastest build (%s) of the unmodified reference: median of %d samples x %.0f s, %d processes (of %d usable cores; best of n/4, n/2, n) "
                          "x %d ch x %d-frame blocks, own 131072-tap IRs; FFT backend = oracle/fftw3_shim.c (FFTW3 absent: pessimistic for the CPU)"
                          % (best, runs, sample_s, procs, ncpu, ch_per_proc, block),
                "channels": procs * ch_per_proc})
    return out


# ------------------------------------------------------------------------------------------------
# device-resident timing of one chain: CUDA events on the launching stream, region closed over all streams
# ------------------------------------------------------------------------------------------------
def time_device(chain, d_in, d_out_ptr, frames, steps, warm, stream, barrier=None):
    """-> (milliseconds for `steps` calls after `warm` untimed ones, kernels launched inside the timed region).
    d_in: list of device tensors (rotating)."""
    import torch
    import dsp_b200
    n = len(d_in)
    for i in range(warm):
        chain.run_device(0, frames, d_in[i % n].data_ptr(), d_out_ptr, stream)
    chain.join(0, stream)
    if barrier:
        barrier()
    else:
        torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = dsp_b200.kernel_launches()
    e0.record()
    for i in range(steps):
        chain.run_device(0, frames, d_in[i % n].data_ptr(), d_out_ptr, stream)
    chain.join(0, stream)            # side-stream work of the timed blocks is inside the region
    e1.record()
    launches = dsp_b200.kernel_launches() - l0
    if barrier:
        barrier()
    else:
        torch.cuda.synchronize()
    return e0.elapsed_time(e1), launches


def fir_bytes_model(plan, C, F, h):
    """Algorithmic HBM bytes per input sample of every kernel of a K2 step (DESIGN.md, K2) from the operator's plan."""
    lv = plan["levels"]
    lvl = lv[-1]
    pf = int(plan.get("tail_pf", 0))
    tb = int(plan.get("t_batch", 0))
    pipe = int(plan.get("pipe", 0))
    ppf = int(plan.get("pipe_pf", 0))
    parts = {}
    P = lvl["P"]
    if pipe:
        # persistent pipeline kernel: in 8, spectrum to the FDL 16, (ppf-1) FDL rows, ppf filter rows, V, carry r/w, out
        parts["fir_pipe"] = 8 + 16 + 16.0 * (ppf - 1) + 16.0 * ppf * h + (16 if tb else 0) + 8 + 8 + 8
        if tb:
            parts["fir_mac_batch"] = 16.0 * ((P - 2 - 1) + (P - 2 - tb) * h + tb) / tb
        return sum(parts.values()), parts
    n_lv = len(lv)
    if pf == 0:
        mac = 16.0 * (P * (1 + h) + 1)
        batch = 0.0
    elif tb:
        # per-block MAC: partitions pf .. pf+tb-1 (a row of X and of H each), V in, Y out.  A batch tier of depth T over
        # n partitions streams n + T - 1 rows of X and n of H once for T block periods, writes T rows of V and -- the
        # near tier of two -- reads the far tier's T rows
        mac = 16.0 * (tb * (1 + h) + 2)
        tf, fe = int(plan.get("t_far", 0)), int(plan.get("far_e", 0))
        n_near = (tf + pf + fe if tf else P) - (tb + pf)
        n_far = P - (tf + pf + fe)
        batch = 16.0 * ((n_near + tb - 1) + n_near * h + tb + (tb if tf else 0)) / tb
        far = 16.0 * ((n_far + tf - 1) + n_far * h + tf) / tf if tf else 0.0
    else:
        mac = 16.0 * ((P - pf) * (1 + h) + 1)
        batch = 0.0
    parts = {"stash_unstash": 0.0, "fir_level0": 0.0, "fir_fwd_inv": 0.0, "fir_mac": mac, "fir_mac_batch": batch}
    if pf and tb and int(plan.get("t_far", 0)):
        parts["fir_mac_batch_far"] = far
    if int(plan.get("merge", 0)):
        # the per-block MAC and the batch launch of the block are one grid
        parts["fir_tail"] = parts.pop("fir_mac") + parts.pop("fir_mac_batch")
    direct = n_lv == 1 and (pf != 0 or P <= 2)
    if not direct:
        parts["stash_unstash"] = 16.0 + (8.0 + 8.0 * (n_lv - 1) + 8.0)
    for i, L in enumerate(lv):
        in_kernel = min(L["P"], 2 if i == 0 else 1)
        has_init = pf and i == n_lv - 1
        if pf == 0 and i == 0 and L["P"] > 2:
            parts["fir_fwd_inv"] += (8 + 16) + (16 + 8 + 8 + 8)
            continue
        parts["fir_level0"] += 8 + 16 + 16 * (in_kernel - 1) + 16 * in_kernel * h + (16 if has_init else 0) + 8 + 8 + 8
    return sum(parts.values()), parts


def eq_coefs(dsp, fs, n):
    return np.array([dsp.biquad_design(13, fs, EQ_F[i], 1.4, EQ_G[i]) for i in range(n)])


def measure_configs(dsp, torch, irs, peak, local_rank, dropin_steps, only=None):
    """Driver-run numbers for the other BASELINE configs (device-resident, 200 blocks each after 5 warm-ups) and for
    the drop-in call path.  Every entry: Msamples/s in, ms per block, and the roofline fraction of its bound."""
    out = {}
    stream = torch.cuda.current_stream().cuda_stream
    steps, warm = 200, 5

    def want(name):
        return not only or name in only

    def entry(name, chain, C, F, fs, bytes_per_sample, extra=None, out_frames=None, note=None):
        d_in = [torch.from_numpy(make_block(F, C, 500 + i)).cuda() for i in range(4)]
        of = out_frames or F
        d_out = torch.empty((of + 8, C), dtype=torch.float64, device="cuda")
        ms, _ = time_device(chain, d_in, d_out.data_ptr(), F, steps, warm, stream)
        rate = C * F * steps / (ms * 1e-3)
        e = {"workload": name, "value": rate / 1e6, "unit": UNIT, "ms_per_block": ms / steps, "blocks": steps, "block_frames": F,
             "channels": C, "fs": fs,
             "roofline": {"bound": "hbm", "algorithmic_bytes_per_sample": bytes_per_sample, "achieved": bytes_per_sample * rate / 1e9,
                          "peak": peak, "unit": "GB/s", "frac": bytes_per_sample * rate / 1e9 / peak}}
        if extra:
            e.update(extra)
        if note:
            e["note"] = note
        chain.close()
        del d_in, d_out
        return e

    # C2: 10-stage eq cascade, 256 ch, 4096-frame blocks (K1: one read + one write of the block)
    C, F = 256, 4096
    if want("C2"):
        ch = dsp.Chain(FS, C, devices=[local_rank]).add_biquad(eq_coefs(dsp, FS, 10))
        out["C2"] = entry("10 x eq cascade, 256 ch, 48 kHz, 4096-frame blocks", ch, C, F, FS, 16.0,
                          note="K1 fused cascade; FP64-issue/latency-bound, HBM bound is 16 B/sample")
    # C3: fir_p 131072 taps, 64 channels
    if want("C3"):
        C = 64
        ch = dsp.Chain(FS, C, devices=[local_rank]).add_fir(irs[:, :C], block_hint=F)
        plan = [op for op in ch.describe() if op.get("op") == "fir"][0]
        bps, _ = fir_bytes_model(plan, C, F, 1)
        out["C3"] = entry("fir_p 131072 taps x 64 ch, per-channel IR, 4096-frame blocks", ch, C, F, FS, bps, extra={"plan": plan})
    # H at the CLI's default block (dsp.h:38).  This shape's step time varies from one chain to the next (61.6 us per
    # block in most, up to 2x that in some: DESIGN.md K2): three fresh chains, the median one is the entry, all three
    # are listed
    if want("H_2048"):
        C, F2 = 256, 2048
        runs = []
        for rep_i in range(3):
            ch = dsp.Chain(FS, C, devices=[local_rank]).add_fir(irs[:, :C], block_hint=F2)
            plan = [op for op in ch.describe() if op.get("op") == "fir"][0]
            bps, _ = fir_bytes_model(plan, C, F2, 1)
            runs.append(entry("fir_p 131072 taps x 256 ch, per-channel IR, 2048-frame blocks (CLI default)", ch, C, F2, FS, bps, extra={"plan": plan}))
        runs.sort(key=lambda e: e["ms_per_block"])
        out["H_2048"] = dict(runs[1], runs_ms_per_block=[e["ms_per_block"] for e in runs],
                             note="median of three fresh chains of 200 blocks each")
    # C4: resample 44100 -> 48000, 1024 ch
    fs4 = 44100
    if want("C4"):
        C = 1024
        ch = dsp.Chain(fs4, C, devices=[local_rank]).add_resample(48000)
        of = ch.max_out_frames(F)
        rp = dsp.resample_params(fs4, 48000)
        flop_per_in = 2.0 * rp["taps_per_phase"] * rp["n"] / rp["d"]
        e = entry("resample 44100 -> 48000, 1024 ch, 4096-frame blocks", ch, C, F, fs4, 8.0 * (1 + rp["n"] / rp["d"]), out_frames=of)
        e["fp64"] = {"flop_per_input_sample": flop_per_in, "achieved_tflops": flop_per_in * e["value"] * 1e6 / 1e12,
                     "fp64_tflops_measured": 37.1, "fp64_peak_source": "scripts/micro/dmma_probe.cu on this pool's B200 (round 1)",
                     "frac_of_fp64_peak": flop_per_in * e["value"] * 1e6 / 1e12 / 37.1}
        e["note"] = "polyphase form as north_star words it: FP64-tensor-core (DMMA) bound, not HBM bound"
        out["C4"] = e
    # C5 share: 8 eq + fir_p 65536 (shared IR) + resample, 256 ch at 44100
    if want("C5_share"):
        C = 256
        h5 = make_ir(65536, 0)
        ch = dsp.Chain(fs4, C, devices=[local_rank]).add_biquad(eq_coefs(dsp, fs4, 8)).add_fir(h5, block_hint=F).add_resample(48000)
        plan = [op for op in ch.describe() if op.get("op") == "fir"][0]
        bps, _ = fir_bytes_model(plan, C, F, 0)
        of = ch.max_out_frames(F)
        out["C5_share"] = entry("8 x eq + fir_p 65536 taps (shared IR) + resample 44100 -> 48000, 256 ch (one GPU's share of config 5)", ch, C, F,
                                fs4, 16.0 + bps + 8.0 * (1 + 160.0 / 147.0), out_frames=of, extra={"plan": plan})
    if not want("dropin"):
        return out

    # e2e_dropin: run_effects_chain() of the reference chain runtime with the shim's GPU effects (shim/frontend.c)
    try:
        from dsp_b200 import frontend
        if frontend.available():
            C, F = 256, 4096
            tmp = tempfile.mkdtemp(prefix="dspb200_dropin_")
            ir_path = os.path.join(tmp, "ir.f64")
            np.ascontiguousarray(irs[:, :C], dtype="<f8").tofile(ir_path)
            pool = np.stack([make_block(F, C, 700 + i) for i in range(4)])
            dd = {}
            for label, pin in (("pageable", None), ("pinned", "1")):
                if pin:
                    os.environ["DSP_B200_PIN"] = pin
                else:
                    os.environ.pop("DSP_B200_PIN", None)
                fc = frontend.DropinChain("fir_p -t pcm -e double -c %d -r %d %s" % (C, FS, ir_path), FS, C)
                sec, f, chk = fc.time(pool, 5, dropin_steps)
                dd[label] = {"value": C * F * dropin_steps / sec / 1e6, "unit": UNIT, "ms_per_block": sec / dropin_steps * 1e3,
                             "blocks": dropin_steps, "effects": fc.effect_names(), "checksum": chk,
                             "buffers": "the frontend's calloc block buffers" + (", page-locked once by the shim (DSP_B200_PIN=1)" if pin else ", pageable")}
                fc.close()
            os.environ.pop("DSP_B200_PIN", None)
            os.remove(ir_path)
            os.rmdir(tmp)
            dd["api"] = "run_effects_chain() (reference effects_chain.c, unmodified) -> shim effect->run() -> dspb200_chain_run_host, in place; clock_gettime around each call"
            dd["workload"] = "fir_p 131072 taps x 256 ch, 4096-frame blocks (the headline through the drop-in)"
            out["e2e_dropin"] = dd
            # config 5's chain through the drop-in: eight eq + fir_p 65536 (shared IR) + resample -- the optimizer merges the
            # same-rate effects, the device hand-off carries the block across the rate change: one device chain per block
            tmp = tempfile.mkdtemp(prefix="dspb200_dropin_")
            ir_path = os.path.join(tmp, "ir5.f64")
            make_ir(65536, 0).astype("<f8").tofile(ir_path)
            eqs = " ".join("eq %g 1.4 %g" % (EQ_F[i], EQ_G[i]) for i in range(8))
            chain5 = "%s fir_p -t pcm -e double -c 1 -r 44100 %s resample 48k" % (eqs, ir_path)
            os.environ["DSP_B200_PIN"] = "1"
            fc = frontend.DropinChain(chain5, 44100, C)
            h0, d0 = dsp.copy_counts()
            sec, f, chk = fc.time(pool, 5, dropin_steps)
            h1, d1 = dsp.copy_counts()
            out["C5_dropin"] = {"workload": "8 x eq + fir_p 65536 (shared IR) + resample 44100 -> 48000, 256 ch, 4096-frame blocks, run_effects_chain() through the drop-in",
                                "value": C * F * dropin_steps / sec / 1e6, "unit": UNIT, "ms_per_block": sec / dropin_steps * 1e3, "blocks": dropin_steps,
                                "effects": fc.effect_names(), "h2d_copies_per_block": (h1 - h0) / float(dropin_steps + 5),
                                "d2h_copies_per_block": (d1 - d0) / float(dropin_steps + 5),
                                "note": "copies are counted per channel slab (4 slabs at 256 channels): one copy in and one out per slab and block = one device chain across the rate change",
                                "checksum": chk}
            fc.close()
            os.environ.pop("DSP_B200_PIN", None)
            os.remove(ir_path)
            os.rmdir(tmp)
        else:
            out["e2e_dropin"] = {"unavailable": "shim/_build/libdsp_b200_frontend.so not built (needs the reference sources at build time)"}
    except Exception as ex:                                            # a failing side measurement must not sink the headline
        out["e2e_dropin"] = {"error": str(ex)[:200]}
    return out


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--block", type=int, default=4096)
    ap.add_argument("--channels", type=int, default=CHANNELS_PER_GPU, help="channels per GPU")
    ap.add_argument("--taps", type=int, default=TAPS)
    ap.add_argument("--shared-ir", action="store_true", help="one IR for all channels (-c 1) instead of one per channel")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--only-configs", default="", help="comma list out of C2,C3,H_2048,C4,C5_share,dropin (measurements)")
    ap.add_argument("--no-kernels", action="store_true", help="skip the per-kernel (serialised) timing pass")
    ap.add_argument("--e2e-slabs", type=int, default=4, help="channel slabs of the synchronous host call (copy-in / kernels / copy-out of the slabs overlap)")
    ap.add_argument("--e2e-pipe-slabs", type=int, default=0, help="channel slabs with blocks in flight (0: same as --e2e-slabs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's output of the headline and e2e paths as DIR/<name>.npy (device, host, host_pipelined)")
    a = ap.parse_args()

    # stdout carries exactly one JSON line: whatever libraries print there (NCCL's version banner under
    # NCCL_DEBUG=VERSION, for one) is sent to stderr, the line itself goes to the saved descriptor
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    def emit(obj):
        real_stdout.write(json.dumps(obj) + "\n")
        real_stdout.flush()

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    steps, warm = max(1, a.steps), max(3, a.warmup)
    config = {"workload": "fir_p %d taps x %d ch per GPU, %s IR, %d-frame blocks, fs %d" %
                          (a.taps, a.channels, "shared" if a.shared_ir else "per-channel", a.block, FS),
              "block_frames": a.block, "channels_per_gpu": a.channels, "taps": a.taps,
              "parallelism": "channel-sharded x%d, no collective" % max(world, 1)}

    if a.impl == "reference":
        if rank != 0:
            return 0
        r = cpu_reference_suite(a.block)
        if r is None:
            emit({"impl": "reference", "unavailable": "oracle/_ref/libdspref.so not built (needs /root/reference at build time)"})
            return 0
        ms_step = r["channels"] * a.block / (r["value"] * 1e6) * 1e3        # one step = one block of every process's channels
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": a.gpus, "steps": steps,
                "warmup": warm, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
                "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "flavour", "spread", "flavours", "cores_usable",
                                                   "cores_os", "process_count_trials_Msps", "process_count_finals_Msps")},
                "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0,
                "note": "time-bounded samples (the reference's fir_p defers work to threads: a fixed handful of blocks reads too fast); "
                        "--steps/--warmup are echoed, the samples are 3 x 5 s per build flavour"}
        emit(line)
        return 0

    os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # one hardware queue per stream of every chain this process builds (before CUDA starts)
    import torch
    import dsp_b200
    from dsp_b200.dist import Job
    if dsp_b200.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device (the product has no CPU path)")
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa(local_rank)      # before any pinned allocation
    job = Job()                      # NCCL process group when WORLD_SIZE > 1: barrier + scalar reductions only
    barrier, reduce_max, reduce_sum = job.barrier, job.reduce_max, job.reduce_sum

    C, F = a.channels, a.block
    irs = make_ir(a.taps, 0)[:, None] if a.shared_ir else make_irs(a.taps, C, first_channel=rank * C)
    n_pool = 8
    blocks = [make_block(F, C, rank * 100 + i) for i in range(n_pool)]

    # ---------------- mode D: device-resident blocks, CUDA events on the launching stream ------------
    chain = dsp_b200.Chain(FS, C, devices=[local_rank]).add_fir(irs, block_hint=F)
    d_blocks = [torch.from_numpy(b).cuda() for b in blocks]
    d_out = torch.empty((F, C), dtype=torch.float64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms, launches = time_device(chain, d_blocks, d_out.data_ptr(), F, steps, warm, stream, barrier=barrier)
    ms = reduce_max(ms)
    total_samples = float(world) * C * F * steps
    value = total_samples / (ms * 1e-3) / 1e6
    checksum = float(d_out.abs().sum().item())
    outputs = {"device": d_out.cpu().numpy()} if a.dump_outputs else {}     # before the per-kernel pass reuses d_out

    plan = [op for op in chain.describe() if op.get("op") == "fir"][0]
    h = 0 if a.shared_ir else 1
    per_sample, parts = fir_bytes_model(plan, C, F, h)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    traffic = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        key = "step:C%d:F%d:taps%d:h%d:pipe%d:far%d" % (C, F, a.taps, h, int(plan.get("pipe", 0)), int(plan.get("t_far", 0)))
        traffic = tr.get(key, {}).get("dram_bytes_per_step")
    except Exception:
        pass
    step_s = ms / steps * 1e-3
    ach = per_sample * C * F / step_s / 1e9
    knames = ("fir_pipe", "fir_level0", "fir_tail", "fir_mac", "fir_mac_batch", "fir_mac_batch_far", "fir_fwd", "fir_inv", "fir_mac_head", "fir_mac_bulk")
    roofline = {"bound": "hbm",
                "kernel": "one step = every kernel of the chain for one block, the look-ahead MACs on their own streams",
                "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                "algorithmic_bytes_per_step": per_sample * C * F, "algorithmic_bytes_per_sample": per_sample,
                "bytes_per_sample_by_kernel": parts, "avg_step_us": step_s * 1e6,
                "plan": plan,
                "note": "achieved = algorithmic bytes of all kernels of a step / measured step time; the timed region ends after "
                        "dspb200_chain_join (every stream of the chain).  `kernels`: each kernel timed alone (side streams folded "
                        "into the caller's stream, profiling events on), outside the headline region."}
    # per-kernel durations: a separate pass with the side streams folded into the caller's stream and event brackets on
    if not a.no_kernels:
        iso = {}
        dsp_b200.debug_serialize(True)
        for i in range(16):
            chain.run_device(0, F, d_blocks[i % n_pool].data_ptr(), d_out.data_ptr(), stream)
        torch.cuda.synchronize()
        for nme in knames:
            dsp_b200.profile_read(nme)
        dsp_b200.profile_enable(True)
        n_iso = 64
        for i in range(n_iso):
            chain.run_device(0, F, d_blocks[i % n_pool].data_ptr(), d_out.data_ptr(), stream)
        torch.cuda.synchronize()
        dsp_b200.profile_enable(False)
        dsp_b200.debug_serialize(False)
        kern = {}
        nB = C * plan["levels"][-1]["B"]
        for nme in knames:
            t_ms, n_l = dsp_b200.profile_read(nme)
            if not n_l:
                continue
            per_launch = parts.get(nme)
            e = {"launches_per_step": n_l / float(n_iso), "alone_us": t_ms / n_l * 1e3}
            if per_launch:
                # bytes_per_sample_by_kernel is per input sample; a launch of the batch kernel covers t_batch block periods
                # (staggered: a launch covers 1/T of the channels for T periods = one block period's share)
                depth = {"fir_mac_batch": plan.get("t_batch", 1), "fir_mac_batch_far": plan.get("t_far", 1)}.get(nme, 1)
                mult = 1 if plan.get("stagger") else depth / max(1, plan.get("far_classes", 1)) if nme == "fir_mac_batch_far" else depth
                e["algorithmic_bytes_per_launch"] = per_launch * nB * mult
                e["alone_GBs"] = e["algorithmic_bytes_per_launch"] / (e["alone_us"] * 1e-6) / 1e9
                e["alone_frac"] = e["alone_GBs"] / peak
            kern["k_" + nme] = e
        roofline["kernels"] = kern
    chain.close()
    del chain

    # ---------------- mode A (e2e): the C-ABI host call on pinned host blocks ------------------------
    e2e = None
    if not a.no_e2e:
        ch2 = dsp_b200.Chain(FS, C, devices=[local_rank], slabs_per_device=a.e2e_slabs).add_fir(irs, block_hint=F)
        pins = [dsp_b200.PinnedArray((F, C), write_combined=True) for _ in range(n_pool)]   # input-only buffers
        for p, b in zip(pins, blocks):
            p.array[:] = b
        pout = dsp_b200.PinnedArray((F, C))
        for i in range(warm):
            ch2.run_raw(F, pins[i % n_pool].ptr, pout.ptr)
        barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            ch2.run_raw(F, pins[i % n_pool].ptr, pout.ptr)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        barrier()
        dt = reduce_max(dt)
        e2e = {"value": total_samples / dt / 1e6, "unit": UNIT, "h2d_bytes_per_step": F * C * 8, "d2h_bytes_per_step": F * C * 8,
               "ms_per_step": dt / steps * 1e3, "api": "dspb200_chain_run_host, pinned host buffers (inputs write-combined), %d channel slabs" % a.e2e_slabs,
               "numa": numa, "checksum": float(np.abs(pout.array).sum())}
        if a.dump_outputs:
            outputs["host"] = pout.array.copy()
        # the same blocks through submit/wait: up to `depth` blocks in flight, each with its own output buffer
        depth = 3
        pslabs = a.e2e_pipe_slabs or a.e2e_slabs
        if pslabs != a.e2e_slabs:
            ch2.close()
            ch2 = dsp_b200.Chain(FS, C, devices=[local_rank], slabs_per_device=pslabs).add_fir(irs, block_hint=F)
        pouts = [dsp_b200.PinnedArray((F, C)) for _ in range(depth + 1)]
        tickets, t_submit, acc = [], 0.0, 0.0
        for i in range(warm):
            ch2.run_raw(F, pins[i % n_pool].ptr, pouts[0].ptr)
        barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            ts = time.perf_counter()
            _, t = ch2.submit_raw(F, pins[i % n_pool].ptr, pouts[i % (depth + 1)].ptr)
            t_submit += time.perf_counter() - ts
            tickets.append(t)
            if i >= depth:
                ch2.wait(tickets[i - depth])
                acc += float(pouts[(i - depth) % (depth + 1)].array[0, 0])     # the block is on the host now
        for t in tickets[-depth:]:
            ch2.wait(t)
        torch.cuda.synchronize()
        dtp = time.perf_counter() - t0
        barrier()
        dtp = reduce_max(dtp)
        e2e["pipelined"] = {"value": total_samples / dtp / 1e6, "unit": UNIT, "ms_per_step": dtp / steps * 1e3,
                            "host_submit_ms_per_step": t_submit / steps * 1e3, "blocks_in_flight": depth, "channel_slabs": pslabs,
                            "api": "dspb200_chain_submit_host + dspb200_chain_wait (same copies, same kernels; the synchronous call above is what the drop-in effect->run() uses)",
                            "checksum": float(np.abs(pouts[(steps - 1) % (depth + 1)].array).sum())}
        if a.dump_outputs:
            outputs["host_pipelined"] = pouts[(steps - 1) % (depth + 1)].array.copy()
        ch2.close()

    clocks = sampler.stop()          # sampled across both timed loops (device-resident and host-call)
    launches_total = int(reduce_sum(float(launches)))
    if outputs and rank == 0:
        dump_outputs(a.dump_outputs, outputs)

    configs = None
    if rank == 0 and world == 1 and not a.no_configs:
        try:
            configs = measure_configs(dsp_b200, torch, irs if not a.shared_ir else make_irs(a.taps, C), peak, local_rank, dropin_steps=100,
                                        only=[v for v in a.only_configs.split(",") if v] or None)
        except Exception as ex:
            configs = {"error": str(ex)[:300]}

    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu:
        r = cpu_reference_suite(F)
        if r:
            cpu = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "flavour", "spread", "flavours", "cores_usable", "cores_os",
                                     "process_count_trials_Msps", "process_count_finals_Msps")}

    if rank == 0:
        config["l2"] = "per-step working set %.2f GB of FDL+filter spectra streamed from HBM (> 126 MB L2); %d rotating input blocks" % (per_sample * C * F / 1e9, n_pool)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warm,
                "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic", "config": config, "clocks": clocks, "e2e": e2e,
                "gpu_launches": launches_total, "roofline": roofline, "cpu_baseline": cpu, "configs": configs, "checksum": checksum}
        emit(line)
    job.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
