#!/usr/bin/env python
"""bench.py -- the WORLD analysis hot path on N B200s (driver contract, see DESIGN.md "Measurement").

One "step" = one pass of {Harvest -> CheapTrick -> D4C} over one batch of synthetic 16 kHz speech
(default: BASELINE.json configs[2], 1024 utterances x 10 s per GPU; weak scaling over ranks with
one NCCL all-gather per output array to reassemble the batch, north_star).  Prints ONE JSON line.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--f0 harvest|dio] [--utts U] [--seconds S] [--fs FS]

value      frames/s with inputs and outputs resident in HBM (CUDA events, max over ranks)
e2e        the same through world_b200_analyze_host(): pinned HOST buffers in, HOST buffers out
roofline   dominant kernel (largest share of the step, timed live with CUDA events inside the
           library): algorithmic HBM bytes / kernel time vs the measured copy peak
cpu_baseline   the compiled reference (oracle/_ref) on this box's host, one thread, bounded sample
--impl reference   the reference's own CPU implementation on all host cores (rank 0 only)
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))



def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--f0", default="harvest", choices=["harvest", "dio"])
    ap.add_argument("--utts", type=int, default=1024, help="utterances per GPU")
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--fs", type=int, default=16000)
    ap.add_argument("--cpu-utts", type=int, default=8, help="utterances of the cpu_baseline sample")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-coded", action="store_true", help="skip the int16-in / coded-out variant of the e2e leg")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-gather", action="store_true")
    ap.add_argument("--reserve-gb", type=float, default=0.0,
                    help="test hook: hold this much extra device memory (emulates the gathered arrays of a larger world)")
    ap.add_argument("--config", type=int, default=0, choices=[0, 2, 3, 4, 5],
                    help="BASELINE.json configs[N-1]: 2 = 1024x10s Dio+StoneMask chain, 3 = 1024x10s Harvest chain (default), "
                         "4 = 256x30s @48 kHz CheapTrick+D4C on a precomputed f0, 5 = 8192x5s Harvest chain sharded over --gpus")
    ap.add_argument("--stages", default="full", choices=["full", "spectral"],
                    help="spectral: time CheapTrick+D4C only, on an f0 computed (untimed) by Dio+StoneMask")
    ap.add_argument("--parity-utts", type=int, default=3, help="extra utterances (middle / last rows of the batch) checked against the reference")
    ap.add_argument("--no-lanes", action="store_true",
                    help="device-resident leg through the separate stage calls on one stream instead of world_b200_analyze_batch")
    ap.add_argument("--slices", type=int, default=1,
                    help="utterance slices per step: F0 of slice s+1 overlaps CheapTrick/D4C of slice s on a second stream")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0) to DIR/<name>.npy, float64, for comparing builds")
    a = ap.parse_args()
    if a.config == 2:
        a.f0, a.utts, a.seconds, a.fs = "dio", 1024, 10.0, 16000
    elif a.config == 3:
        a.f0, a.utts, a.seconds, a.fs = "harvest", 1024, 10.0, 16000
    elif a.config == 4:
        a.f0, a.utts, a.seconds, a.fs, a.stages = "dio", 256, 30.0, 48000, "spectral"
    elif a.config == 5:
        a.f0, a.utts, a.seconds, a.fs = "harvest", max(1, 8192 // max(1, a.gpus)), 5.0, 16000
    return a


def chain_name(a):
    if a.stages == "spectral":
        return "CheapTrick+D4C"
    return "Harvest+CheapTrick+D4C" if a.f0 == "harvest" else "Dio+StoneMask+CheapTrick+D4C"


def workload_name(a):
    tail = " (f0 from Dio+StoneMask, not timed)" if a.stages == "spectral" else ""
    return f"{a.utts}x{a.seconds:g}s synthetic {a.fs // 1000} kHz batch per GPU, {chain_name(a)}{tail}"


def metric_name(a):
    return f"analysis frames/sec ({chain_name(a)})"


def ref_chain(ref, a, xu, keep=False):
    """The reference's own chain on one utterance (oracle/_ref, stock API).  Returns frames, or all outputs."""
    import numpy as np
    xu = np.ascontiguousarray(xu)
    if a.f0 == "harvest":
        t, f0 = ref.harvest(xu, a.fs)
    else:
        t, f0 = ref.dio(xu, a.fs)
        f0 = ref.stonemask(xu, a.fs, t, f0)
    opt = ref.cheaptrick_option(a.fs)
    sp = ref.cheaptrick(xu, a.fs, t, f0, opt)
    ap = ref.d4c(xu, a.fs, t, f0, opt.fft_size)
    return (t, f0, sp, ap) if keep else len(f0)


def parity_entry(np, got, want):
    """got / want: (time_axis, f0, sp, ap) of one utterance.  Relative errors against the reference; entries
    where the reference is exactly 0 must be exactly 0."""
    def rel(g, w):
        den = np.where(w == 0, 1.0, np.abs(w))
        return np.abs(g - w) / den
    t, f0, sp, ap = got
    tr, fr, spr, apr = want
    flips = int(((f0 > 0) != (fr > 0)).sum())
    both = (f0 > 0) & (fr > 0)
    e = {"time_axis_exact": bool(np.array_equal(t, tr)), "frames": int(len(fr)), "vuv_flips": flips,
         "f0_max_rel": float(rel(f0[both], fr[both]).max()) if both.any() else 0.0}
    for name, g, w in (("sp", sp, spr), ("ap", ap, apr)):
        r = rel(g, w)
        e[name + "_max_rel"] = float(r.max())
        e[name + "_frac_gt_1e-6"] = float((r > 1e-6).mean())
    return e


def parity_summary(entries, rows, what):
    if not entries:
        return None
    keys = ["f0_max_rel", "sp_max_rel", "ap_max_rel", "sp_frac_gt_1e-6", "ap_frac_gt_1e-6"]
    out = {"against": what, "rows": rows, "frames": sum(e["frames"] for e in entries),
           "time_axis_bit_exact": all(e["time_axis_exact"] for e in entries),
           "vuv_flips": sum(e["vuv_flips"] for e in entries)}
    for k in keys:
        out[k] = max(e[k] for e in entries)
    out["within_1e-6"] = bool(out["time_axis_bit_exact"] and out["vuv_flips"] == 0 and
                              max(out["f0_max_rel"], out["sp_max_rel"], out["ap_max_rel"]) <= 1e-6)
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dump_outputs(d, arrays, budget=60_000_000, seed=0):
    """arrays: name -> [U, L, ...] tensor of one step (L frames).  The f0 contours of every utterance (if they take at
    most half the budget); of every array, the same fixed seeded sample of utterance rows, as many as fit in what is
    left, and where not even one row fits, of that row a fixed seeded sample of frames (first and last included).
    The row and frame indices go to rows.npy and frames.npy.  Returns them."""
    import numpy as np
    import torch
    os.makedirs(d, exist_ok=True)
    U, L = arrays["f0"].shape
    full_f0 = arrays["f0"].numel() * 8 <= budget // 2
    left = budget - (arrays["f0"].numel() * 8 if full_f0 else 0)
    per_frame = sum(a[0, 0].numel() * 8 for a in arrays.values())
    rng = np.random.default_rng(seed)
    k = max(1, min(U, left // (per_frame * L)))
    rows = np.sort(rng.choice(U, size=k, replace=False))
    frames = np.arange(L)
    if left < per_frame * L:
        inner = rng.choice(np.arange(1, L - 1), size=max(0, left // per_frame - 2), replace=False)
        frames = np.sort(np.concatenate([[0, L - 1], inner]))
    dev = arrays["f0"].device
    ri, fi = torch.as_tensor(rows, device=dev), torch.as_tensor(frames, device=dev)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), a.index_select(0, ri).index_select(1, fi).double().cpu().numpy())
    if full_f0:
        np.save(os.path.join(d, "f0_all.npy"), arrays["f0"].double().cpu().numpy())
    np.save(os.path.join(d, "rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(d, "frames.npy"), frames.astype(np.float64))
    return {"rows": rows.tolist(), "frames": int(len(frames)), "frames_of": int(L)}


def frames_of(fs, n_samples, frame_period=5.0):
    return int(1000.0 * n_samples / fs / frame_period) + 1


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def algorithmic_bytes_per_step(kernel, a, n_utts):
    """Compulsory HBM bytes one step moves through `kernel` (DESIGN.md "Kernels", SURVEY.md 8d)."""
    fs = a.fs
    n = int(a.fs * a.seconds)
    L = frames_of(fs, n)
    L1 = frames_of(fs, n, 1.0)
    fft = 2 ** (1 + int(math.log(3.0 * fs / 71.0 + 1) / math.log(2.0)))
    bins = fft // 2 + 1
    hop = 8 * (fs * 5 // 1000)
    ratio = max(1, int(fs / 8000.0 + 0.5))
    ylen = math.ceil(n / ratio)
    table = {
        # waveform hop once + one output row per frame (SURVEY.md 8d: 4744 B/frame @16 kHz)
        "ct_frame_kernel": n_utts * L * (hop + 8 * bins),
        "d4c_body_kernel": n_utts * L * (hop + 8 * bins),
        "d4c_lovetrain_kernel": n_utts * L * (hop + 16),
        # decimated waveform once + the candidate map it produces (152 channels x 1 ms frames)
        "band_sweep_kernel": n_utts * (ylen * 8 + (152 if a.f0 == "harvest" else 7) * (L1 if a.f0 == "harvest" else L) * 8),
        "band_sweep_ripple_kernel": n_utts * (ylen * 8 + (152 if a.f0 == "harvest" else 7) * (L1 if a.f0 == "harvest" else L) * 8),
        # split sweep: decimated waveform once per band (L2 hits) + complete edge lists out; lists in, candidate map out
        "band_fir_events_kernel": n_utts * (ylen * 8 + 152 * L1 * 8),
        "band_interp_kernel": n_utts * 152 * L1 * 8,
        "band_sweep_list_kernel": 0,
        "harvest_refine_chain_o5_kernel": n_utts * (ylen * 8 + L1 * 21 * 16),
        "d4c_body_slow_kernel": 0,
        "nyquist_bins_kernel": n_utts * ylen * 8,
        "harvest_refine_chain_kernel": n_utts * (ylen * 8 + L1 * 21 * 16),
        # candidate map in, refined candidates + scores out (upper bound 105 slots)
        "harvest_refine_kernel": n_utts * (ylen * 8 + L1 * 21 * 16),
        "harvest_detect_kernel": n_utts * 152 * L1 * 8,
        "harvest_remove_kernel": n_utts * L1 * 21 * 32,
        "harvest_contour_kernel": n_utts * L1 * 21 * 16,
        "harvest_smooth_kernel": n_utts * L1 * 16,
        "harvest_prep_kernel": n_utts * n * 8 * 2,
        "rng_fill_kernel": 0,
        "stonemask_kernel": n_utts * L * (hop + 16),
        "fir_plain_kernel": n_utts * n * 16,
    }
    return table.get(kernel)


_REF = None


def _ref_worker_init(cores_list, counter):
    """One process per host core, pinned: the reference news / frees an FFT plan ~182 k times per utterance
    (harvest.cpp:545-546); threads of one process serialise on the glibc arena, processes do not."""
    global _REF
    with counter.get_lock():
        idx = counter.value
        counter.value += 1
    try:
        os.sched_setaffinity(0, {cores_list[idx % len(cores_list)]})
    except Exception:
        pass
    import torch
    torch.set_num_threads(1)
    from refworld import RefWorld, REF_LIB, ORACLE_LIB
    _REF = RefWorld(REF_LIB if os.path.exists(REF_LIB) else ORACLE_LIB)


_REF_X = {}


def _ref_worker_run(args):
    a, seed = args
    x = _REF_X[seed]     # generated by the parent before the fork: resident, shared copy-on-write
    t0 = time.perf_counter()
    if a.stages == "spectral":
        t, f0 = _REF.dio(x, a.fs)
        f0 = _REF.stonemask(x, a.fs, t, f0)
        t0 = time.perf_counter()     # the f0 stage is not part of this workload
        opt = _REF.cheaptrick_option(a.fs)
        _REF.cheaptrick(x, a.fs, t, f0, opt)
        _REF.d4c(x, a.fs, t, f0, opt.fft_size)
        frames = len(f0)
    else:
        frames = ref_chain(_REF, a, x)
    return frames, time.perf_counter() - t0


def run_reference(a, rank, world):
    """--impl reference: the unmodified reference (oracle/_ref) on all host cores, rank 0 only.  One pinned worker
    process per core; a step = one utterance of the named workload per core (a bounded sample of the batch)."""
    if rank != 0:
        return
    import multiprocessing as mp
    from refworld import REF_LIB
    try:
        cores_list = sorted(os.sched_getaffinity(0))
    except Exception:
        cores_list = list(range(os.cpu_count() or 1))
    cores = len(cores_list)
    per_step = cores
    from synth import synth_batch
    n = int(a.fs * a.seconds)
    for s0 in range(1, per_step + 1, 16):
        seeds = list(range(s0, min(per_step, s0 + 15) + 1))
        xs = synth_batch(seeds, a.fs, n, device="cpu").numpy()
        for j, sd in enumerate(seeds):
            _REF_X[sd] = xs[j].copy()
    ctx = mp.get_context("fork")
    counter = ctx.Value("i", 0)
    with ctx.Pool(cores, initializer=_ref_worker_init, initargs=(cores_list, counter)) as pool:
        jobs = [(a, s) for s in range(1, per_step + 1)]
        for _ in range(max(1, min(a.warmup, 1))):
            pool.map(_ref_worker_run, jobs, chunksize=1)
        t0 = time.perf_counter()
        frames, busy = 0, 0.0
        for _ in range(a.steps):
            res = pool.map(_ref_worker_run, jobs, chunksize=1)
            frames += sum(r[0] for r in res)
            busy += sum(r[1] for r in res)
        dt = time.perf_counter() - t0
        # single-core figure on an otherwise idle box: the denominator of the parallel efficiency
        f1, t_in = pool.apply(_ref_worker_run, ((a, 1),))
        single = f1 / t_in
    value = frames / dt
    sample = (f"{per_step} utterances x {a.seconds:g} s per step (one pinned process per core, {cores} cores, one utterance each), "
              f"{a.steps} steps; in-worker time {busy / a.steps:.1f} core-s per step")
    out = {"impl": "reference", "metric": metric_name(a), "value": value, "unit": "frames/s", "n_gpus": a.gpus,
           "steps": a.steps, "warmup": a.warmup, "ms_per_step": dt / a.steps * 1e3, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": workload_name(a), "fs": a.fs, "frame_period_ms": 5.0,
                      "sample_per_step": f"{per_step} utterances of the named batch"},
           "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores,
                            "kind": "reference" if os.path.exists(REF_LIB) else "port", "sample": sample,
                            "single_core_value": single, "parallel_efficiency": value / (cores * single)},
           "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


def main():
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        run_reference(a, rank, world)
        return
    import numpy as np
    import torch
    import torch.distributed as dist
    from world_b200.api import World, F0_HARVEST, F0_DIO_STONEMASK
    from synth import synth_batch

    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        # NCCL prints its version banner on stdout when the first communicator is created; the contract
        # is ONE JSON line on stdout, so fd 1 points at stderr until the communicator exists.
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    w = World(device=local)
    if world > 1:
        # the library's own NCCL communicator (C ABI, include/world_b200.h): torch.distributed only carries the 128-byte id
        idt = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(w.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            w.comm_init(world, rank, bytes(idt.cpu().numpy().tobytes()))
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    fs, n = a.fs, int(a.fs * a.seconds)
    U = a.utts
    L = frames_of(fs, n)
    # synthetic batch of this rank (seeds distinct across ranks), built on the device
    x = torch.empty((U, n), dtype=torch.float64, device=dev)
    for u0 in range(0, U, 64):
        u1 = min(U, u0 + 64)
        x[u0:u1] = synth_batch(range(rank * U + u0 + 1, rank * U + u1 + 1), fs, n, device=dev)
    opt = w.cheaptrick_option(fs)
    bins = opt.fft_size // 2 + 1
    # outputs: with N > 1 each rank writes its shard straight into the gathered arrays
    free, total = torch.cuda.mem_get_info(dev)
    gather = world > 1 and not a.no_gather
    need_full = 2 * world * U * L * bins * 8
    gather_full = gather and need_full + (24 << 30) < free
    G = world if gather_full else 1
    sp_all = torch.empty((G * U, L, bins), dtype=torch.float64, device=dev)
    ap_all = torch.empty((G * U, L, bins), dtype=torch.float64, device=dev)
    off = rank * U if gather_full else 0
    sp, ap = sp_all[off:off + U], ap_all[off:off + U]
    f0_all = torch.empty((world * U, L), dtype=torch.float64, device=dev)
    t_all = torch.empty((world * U, L), dtype=torch.float64, device=dev)
    reserve = torch.empty(int(a.reserve_gb * (1 << 30)), dtype=torch.uint8, device=dev) if a.reserve_gb > 0 else None
    # scratch budget follows what is left after the (possibly gathered) outputs are resident
    free_now, _ = torch.cuda.mem_get_info(dev)
    budget = int(min(96 << 30, max(2 << 30, free_now * 0.45)))
    w.set_scratch_budget(budget)

    # Two contexts on two streams: the F0 estimator of slice s+1 (FP64 bound) runs concurrently with
    # CheapTrick + D4C of slice s (shared-memory / barrier bound); slices are contiguous utterance ranges.
    n_slices = max(1, min(a.slices, U))
    w2 = World(device=local) if n_slices > 1 else w
    side = torch.cuda.Stream(device=dev) if n_slices > 1 else None
    bounds = [U * i // n_slices for i in range(n_slices + 1)]
    # this rank's f0 / time axis rows live inside the gathered arrays (in-place all-gather)
    t_loc = t_all[rank * U:(rank + 1) * U] if gather else torch.zeros((U, L), dtype=torch.float64, device=dev)
    f0_loc = f0_all[rank * U:(rank + 1) * U] if gather else torch.zeros((U, L), dtype=torch.float64, device=dev)
    if w2 is not w:
        w2.set_scratch_budget(budget // 2)
        w.set_scratch_budget(budget // 2)

    spectral = a.stages == "spectral"
    if spectral:   # config 4: the f0 contour is an input of the timed region (SURVEY.md 8d config 4)
        t_fix = torch.empty((U, L), dtype=torch.float64, device=dev)
        f0_fix = torch.empty((U, L), dtype=torch.float64, device=dev)
        for u0 in range(0, U, 64):
            u1 = min(U, u0 + 64)
            tt, ff, _ = w.dio(x[u0:u1], fs)
            f0_fix[u0:u1] = w.stonemask(x[u0:u1], fs, tt, ff)
            t_fix[u0:u1] = tt
        w.synchronize()

    use_lanes = not spectral and not a.no_lanes and n_slices == 1
    ao_dev = w.analysis_option(fs, F0_HARVEST if a.f0 == "harvest" else F0_DIO_STONEMASK)

    def step():
        main = torch.cuda.current_stream(dev)
        if use_lanes and gather_full:
            # multi-GPU: the same call with the FULL arrays; every finished slice is broadcast to the other ranks by the
            # library's NCCL communicator while the next slice is computed
            w.analyze_batch_allgather(x, fs, ao_dev, t_all, f0_all, sp_all, ap_all)
        elif use_lanes:   # the whole chain in one C-ABI call: utterance slices on two internal streams
            w.analyze_batch(x, fs, ao_dev, time_axis=t_loc, f0=f0_loc, spectrogram=sp, aperiodicity=ap)
        for si in range(0 if use_lanes else n_slices):
            b0, b1 = bounds[si], bounds[si + 1]
            xs = x[b0:b1]
            if spectral:
                t, f0 = t_fix[b0:b1], f0_fix[b0:b1]
            elif a.f0 == "harvest":
                t, f0, fl = w.harvest(xs, fs)
            else:
                t, f0, fl = w.dio(xs, fs)
                f0 = w.stonemask(xs, fs, t, f0)
            t_loc[b0:b1].copy_(t); f0_loc[b0:b1].copy_(f0)
            if side is None:
                w.cheaptrick(xs, fs, t, f0, opt, out=sp[b0:b1])
                w.d4c(xs, fs, t, f0, opt.fft_size, out=ap[b0:b1])
            else:
                ev = torch.cuda.Event()
                ev.record(main)
                with torch.cuda.stream(side):
                    side.wait_event(ev)
                    t.record_stream(side); f0.record_stream(side)
                    w2.cheaptrick(xs, fs, t, f0, opt, out=sp[b0:b1])
                    w2.d4c(xs, fs, t, f0, opt.fft_size, out=ap[b0:b1])
        if side is not None:
            main.wait_stream(side)
        t, f0 = t_loc, f0_loc
        if gather and not (use_lanes and gather_full):   # in-place all-gathers through the C ABI (wb_multi.cu)
            w.allgather_rows(f0_all, U)
            w.allgather_rows(t_all, U)
            if gather_full:
                w.allgather_rows(sp_all, U)
                w.allgather_rows(ap_all, U)
        return f0

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(a.warmup):
        step()
    barrier()
    w.synchronize()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    w.profile(True)
    launches0 = w.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(a.steps):
        f0_last = step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = w.launch_count() - launches0
    w.profile(False)
    prof = w.profile_report()
    clocks = sampler.stop() if rank == 0 else None
    w.synchronize()
    dumped = None
    if a.dump_outputs and rank == 0:   # what a caller of the timed path receives from its last step
        dumped = dump_outputs(a.dump_outputs, {"time_axis": t_fix if spectral else t_loc, "f0": f0_fix if spectral else f0_loc,
                                               "spectrogram": sp, "aperiodicity": ap})
    if world > 1:
        tms = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms = float(tms.item())
    frames_step = world * U * L
    value = frames_step * a.steps / (ms / 1e3)

    # ---- multi-GPU equality: what another rank contributed to the gathered arrays is bit-identical to what
    # this rank computes for the same utterances on its own GPU (outside the timed region, rank 0 only)
    gather_check = None
    if world > 1 and gather and rank == 0:
        try:
            ok, checked = True, []
            for r in range(1, world):     # the first utterance of EVERY other rank's shard
                xs = synth_batch(range(r * U + 1, r * U + min(U, 64) + 1), fs, n, device=dev)[:1].contiguous()   # same generator call shape as that rank's
                tt, ff, _ = (w.harvest(xs, fs) if a.f0 == "harvest" else w.dio(xs, fs))
                if a.f0 != "harvest":
                    ff = w.stonemask(xs, fs, tt, ff)
                ok = ok and torch.equal(ff, f0_all[r * U:r * U + 1]) and torch.equal(tt, t_all[r * U:r * U + 1])
                if gather_full:
                    ok = ok and torch.equal(w.cheaptrick(xs, fs, tt, ff, opt), sp_all[r * U:r * U + 1])
                    ok = ok and torch.equal(w.d4c(xs, fs, tt, ff, opt.fft_size), ap_all[r * U:r * U + 1])
                checked.append(r * U)
            gather_check = {"bit_identical": bool(ok), "rows": checked}
        except Exception as e:  # never let the check take the bench line down
            gather_check = f"error: {e}"

    # ---- rows of the TIMED batch kept for the parity report (compared with the reference's own chain below)
    k_cpu = 0 if a.no_cpu else max(1, min(a.cpu_utts if world == 1 else 1, U))
    par_rows = list(range(k_cpu))
    for r in ([U // 2 - 1, U // 2, U - 1][:max(0, a.parity_utts)] if not a.no_cpu else []):
        if 0 <= r < U and r not in par_rows:
            par_rows.append(r)
    par_dev = {}
    if rank == 0:
        tsrc, fsrc = (t_fix, f0_fix) if spectral else (t_loc, f0_loc)
        for r in par_rows:
            par_dev[r] = (tsrc[r].cpu().numpy(), fsrc[r].cpu().numpy(), sp[r].cpu().numpy(), ap[r].cpu().numpy())
        par_x = {r: x[r].cpu().numpy() for r in par_rows}
    par_e2e = {}

    # ---- end to end through the host-pointer ABI (pinned host buffers, copies inside the timed region)
    e2e = None
    if not a.no_e2e:
        import psutil
        need = U * n * 8 + 2 * U * L * bins * 8 + 2 * U * L * 8
        avail = psutil.virtual_memory().available
        Ue = U
        while Ue > 16 and need * Ue / U * 1.3 * world > avail:   # every rank of the node pins its own buffers
            Ue //= 2
        xh = torch.empty((Ue, n), dtype=torch.float64, pin_memory=True)
        xh.copy_(x[:Ue])
        th = torch.empty((Ue, L), dtype=torch.float64, pin_memory=True)
        fh = torch.empty((Ue, L), dtype=torch.float64, pin_memory=True)
        sph = torch.empty((Ue, L, bins), dtype=torch.float64, pin_memory=True)
        aph = torch.empty((Ue, L, bins), dtype=torch.float64, pin_memory=True)
        # free the device-resident outputs of the first phase: analyze_host brings its own buffers
        del sp, ap, sp_all, ap_all
        torch.cuda.empty_cache()
        w.trim()   # ... and the scratch arenas the device-resident leg grew (both lanes)
        # the (possibly gathered) outputs are gone: let the pipeline size its chunks for what is free now
        free_e2e, _ = torch.cuda.mem_get_info(dev)
        w.set_scratch_budget(int(min(96 << 30, max(2 << 30, free_e2e * 0.45))))
        ao = w.analysis_option(fs, F0_HARVEST if a.f0 == "harvest" else F0_DIO_STONEMASK)
        if spectral:
            th.copy_(t_fix[:Ue]); fh.copy_(f0_fix[:Ue])
            sub = 32     # utterances per upload / compute / download round
            xd = torch.empty((sub, n), dtype=torch.float64, device=dev)
            td = torch.empty((sub, L), dtype=torch.float64, device=dev)
            fd = torch.empty((sub, L), dtype=torch.float64, device=dev)
            spd = torch.empty((sub, L, bins), dtype=torch.float64, device=dev)
            apd = torch.empty((sub, L, bins), dtype=torch.float64, device=dev)

            def e2e_step():   # host waveform + host f0 in, host spectrogram + aperiodicity out, batched C ABI in between
                for u0 in range(0, Ue, sub):
                    m = min(sub, Ue - u0)
                    xd[:m].copy_(xh[u0:u0 + m], non_blocking=True)
                    td[:m].copy_(th[u0:u0 + m], non_blocking=True)
                    fd[:m].copy_(fh[u0:u0 + m], non_blocking=True)
                    w.cheaptrick(xd[:m], fs, td[:m], fd[:m], opt, out=spd[:m])
                    w.d4c(xd[:m], fs, td[:m], fd[:m], opt.fft_size, out=apd[:m])
                    sph[u0:u0 + m].copy_(spd[:m], non_blocking=True)
                    aph[u0:u0 + m].copy_(apd[:m], non_blocking=True)
                torch.cuda.synchronize()
        else:
            w.lib.world_b200_set_stream(w._h, None)

            def e2e_step():
                w.analyze_host(xh, fs, ao, time_axis=th, f0=fh, spectrogram=sph, aperiodicity=aph, f0_stride=L)

        e2e_step()
        barrier()
        t0 = time.perf_counter()
        ke = max(1, min(a.steps, 3))
        e2e_steps_ms = []
        for _ in range(ke):
            t1 = time.perf_counter()
            e2e_step()
            e2e_steps_ms.append((time.perf_counter() - t1) * 1e3)
        barrier()
        dt = time.perf_counter() - t0
        if world > 1:
            tdt = torch.tensor([dt], dtype=torch.float64, device=dev)
            dist.all_reduce(tdt, op=dist.ReduceOp.MAX)
            dt = float(tdt.item())
        e2e = {"value": world * Ue * L * ke / dt, "unit": "frames/s",
               "h2d_bytes_per_step": int(Ue * n * 8), "d2h_bytes_per_step": int(2 * Ue * L * bins * 8 + 2 * Ue * L * 8),
               "utts_per_gpu": Ue, "steps": ke, "ms_per_step_rank0": e2e_steps_ms,
               "note": ("world_b200_cheaptrick_batch + world_b200_d4c_batch on 32-utterance rounds: pinned host waveform / f0 up, pinned host rows down"
                        if spectral else
                        "world_b200_analyze_host: pinned host buffers in/out; F0 stage on 512-utterance chunks, CheapTrick+D4C on 128-utterance sub-chunks (32 in the last chunk) whose rows are downloaded while the next ones are computed")}
        if spectral:
            e2e["h2d_bytes_per_step"] = int(Ue * n * 8 + 2 * Ue * L * 8)
            e2e["d2h_bytes_per_step"] = int(2 * Ue * L * bins * 8)
        # the e2e result must be the same numbers the device-resident path produced
        same = bool(torch.equal(fh, f0_last[:Ue].cpu()))
        e2e["matches_device_path"] = same
        if rank == 0:
            for r in par_rows:
                if r < Ue:
                    par_e2e[r] = (th[r].numpy().copy(), fh[r].numpy().copy(), sph[r].numpy().copy(), aph[r].numpy().copy())
        # the same chain with the ingest (int16 PCM in) and the codec (60 mel-cepstral dimensions + band
        # aperiodicities out) fused in on the device -- SURVEY.md 8 rows f2/f3: what crosses PCIe shrinks
        if not a.no_coded and not spectral:
            try:
                dims = 60
                n_ap = max(1, w.number_of_aperiodicities(fs))
                del sph, aph
                ph = torch.empty((Ue, n), dtype=torch.int16, pin_memory=True)
                ph.copy_((xh * 32767.0).round().to(torch.int16))
                csh = torch.empty((Ue, L, dims), dtype=torch.float64, pin_memory=True)
                cah = torch.empty((Ue, L, n_ap), dtype=torch.float64, pin_memory=True)

                def coded_step():
                    w.analyze_coded_host(ph, 16, fs, ao, dims, time_axis=th, f0=fh, coded_sp=csh, coded_ap=cah, f0_stride=L)

                coded_step()
                barrier()
                t0 = time.perf_counter()
                for _ in range(ke):
                    coded_step()
                barrier()
                dtc = time.perf_counter() - t0
                if world > 1:
                    tdt = torch.tensor([dtc], dtype=torch.float64, device=dev)
                    dist.all_reduce(tdt, op=dist.ReduceOp.MAX)
                    dtc = float(tdt.item())
                e2e["coded"] = {"value": world * Ue * L * ke / dtc, "unit": "frames/s",
                                "h2d_bytes_per_step": int(Ue * n * 2),
                                "d2h_bytes_per_step": int(Ue * L * (dims + n_ap) * 8 + 2 * Ue * L * 8),
                                "note": "world_b200_analyze_coded_host: int16 PCM in, CodeSpectralEnvelope(60) + "
                                        "CodeAperiodicity rows out, computed in the frame kernels (no full rows in HBM); "
                                        "input is the 16-bit quantisation of the same waveforms"}
            except Exception as exc:   # the secondary leg must never take the bench line down
                e2e["coded"] = {"error": f"{type(exc).__name__}: {exc}"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (timed live above)
    peak, peak_src = measured_peak_hbm()
    kernels = {k: {"ms_per_step": v["ms"] / a.steps, "launches_per_step": v["launches"] / a.steps} for k, v in prof.items()}
    dom = max(kernels, key=lambda k: kernels[k]["ms_per_step"]) if kernels else None
    roof = None
    if dom:
        nbytes = algorithmic_bytes_per_step(dom, a, U)
        kms = kernels[dom]["ms_per_step"]
        achieved = (nbytes / 1e9) / (kms / 1e3) if nbytes else None
        traffic = None
        tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tp):
            per_utt = json.load(open(tp)).get(dom, {}).get("dram_bytes_per_utt")
            if per_utt:
                traffic = per_utt * U / max(1.0, kernels[dom]["launches_per_step"])
        roof = {"kernel": dom, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak if achieved else None, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": nbytes / max(1.0, kernels[dom]["launches_per_step"]) if nbytes else None,
                "kernel_ms_per_step": kms, "share_of_step": kms / (ms / a.steps),
                "note": "FP64-ALU/shared-memory bound path (SURVEY.md 8d): HBM fraction is reported as BASELINE.json asks"}

    # ---- FP64 view of the two FP64-bound kernels (the binding roofline, DESIGN.md 4)
    fp64 = None
    try:
        peak64 = w.fp64_peak()
        ratio = max(1, int(fs / 8000.0 + 0.5))
        ylen = math.ceil(n / ratio)
        fir_flops = None
        if a.f0 == "harvest":
            afs = fs / ratio
            taps = 0
            for i in range(152):
                bnd = 71.0 * 0.9 * 2.0 ** ((i + 1) / 40.0)
                taps += 2 * int(afs / bnd * 2.0 + 0.5) + 1
            fir_flops = 2.0 * taps * ylen * U  # one FMA per tap and output sample
        fp64 = {"peak_tflops": peak64, "peak_source": "world_b200_fp64_peak (8 DFMA chains/thread, CUDA events)"}
        if fir_flops and "band_sweep_kernel" in kernels:
            t_s = kernels["band_sweep_kernel"]["ms_per_step"] / 1e3
            fp64["band_sweep_fir_tflops"] = fir_flops / t_s / 1e12
            fp64["band_sweep_frac"] = fir_flops / t_s / 1e12 / peak64
    except Exception as e:  # never let the extra figure break the bench line
        fp64 = {"error": str(e)[:100]}

    # ---- CPU baseline: the compiled reference, one thread, bounded sample of the same batch; its OUTPUTS are the
    # parity check of the timed batch (rows 0..k-1 plus the middle / last rows: real chunk boundaries and ring sizes)
    cpu, parity = None, None
    if not a.no_cpu:
        from refworld import RefWorld, REF_LIB, ORACLE_LIB
        kind, lib = ("reference", REF_LIB) if os.path.exists(REF_LIB) else ("port", ORACLE_LIB)
        ref = RefWorld(lib)
        want = {}
        t0 = time.perf_counter()
        fr = 0
        dt = None
        for j, r in enumerate(par_rows):
            if j == k_cpu:
                dt = time.perf_counter() - t0
            if spectral:   # the f0 stage is not part of this workload: the reference runs on the same contour
                tr_, fr_ = par_dev[r][0], par_dev[r][1]
                xu = np.ascontiguousarray(par_x[r])
                o = ref.cheaptrick_option(fs)
                want[r] = (tr_, fr_, ref.cheaptrick(xu, fs, tr_, fr_, o), ref.d4c(xu, fs, tr_, fr_, o.fft_size))
            else:
                want[r] = ref_chain(ref, a, par_x[r], keep=True)
            if j < k_cpu:
                fr += len(want[r][1])
        if dt is None:
            dt = time.perf_counter() - t0
        if world == 1:
            cpu = {"value": fr / dt, "unit": "frames/s", "cores": 1, "kind": kind,
                   "sample": f"utterances 1..{k_cpu} of the batch ({k_cpu} x {a.seconds:g} s), single thread, {dt:.1f} s",
                   "host_cores_available": os.cpu_count()}
        what = ("the reference's own chain (oracle/_ref: its f0 -> its CheapTrick / D4C) on the same waveforms" if not spectral
                else "oracle/_ref CheapTrick / D4C on the same waveforms and f0 contour")
        parity = {"device_resident": parity_summary([parity_entry(np, par_dev[r], want[r]) for r in par_rows], par_rows, what),
                  "e2e_host_arrays": parity_summary([parity_entry(np, par_e2e[r], want[r]) for r in par_rows if r in par_e2e],
                                                    [r for r in par_rows if r in par_e2e], what),
                  "tolerance": "1e-6 relative (north_star); time_axis bit exact; no V/UV flip"}

    out = {"metric": metric_name(a),
           "value": value, "unit": "frames/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
           "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f64", "data": "synthetic",
           "config": {"workload": workload_name(a), "baseline_config": a.config or None, "fs": fs, "frame_period_ms": 5.0, "frames_per_step": frames_step,
                      "l2_policy": "inputs+outputs per step (>= 18 GB) exceed the 126 MB L2; no flush needed",
                      "multi_gpu": ("utterances sharded over ranks; the library's own NCCL communicator (C ABI) reassembles f0/time_axis" +
                                    ("/spectrogram/aperiodicity, slice by slice under the compute (peer-to-peer copies over CUDA IPC mappings; NCCL broadcasts with WB_NO_P2P=1)" if gather_full else "")) if world > 1 else "single GPU",
                      "gathered_equals_local_recompute": gather_check},
           "clocks": clocks, "e2e": e2e, "slices": n_slices,
           "device_resident_api": ("world_b200_analyze_batch (utterance slices on two internal streams; per-kernel times below overlap, "
                                   "their sum exceeds the step)" if use_lanes else "separate *_batch stage calls on one stream"), "gpu_launches": int(launches), "roofline": roof, "fp64": fp64, "cpu_baseline": cpu,
           "parity": parity, "kernels": kernels}
    if dumped is not None:
        out["dumped"] = dumped
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
