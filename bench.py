#!/usr/bin/env python
"""bench.py -- Mpix/s advected on BASELINE.json's config[1]:
2048x2048 synthetic radar frames, motion field + 12-leadtime semi-Lagrangian
extrapolation.

    python bench.py --gpus N --steps K --warmup W          (ours, CUDA)
    python bench.py --impl reference ...                   (CPU oracle port, all host cores)

Headline (every N): one "step" = one pass of the hot path over one batch of synthetic input, on
every rank:
  motion field from this rank's last two frames (dense Lucas-Kanade),
  12-leadtime semi-Lagrangian extrapolation of this rank's field with it.
Metric: Mpix/s advected = (N * T * m * n) / step time, max over ranks (weak scaling: N
independent nowcasts, one per GPU, no collective on the data path).

The same JSON line carries two more blocks, measured at every N with the same timing rules
(`--no-extras` skips them, `--workload X` makes X the headline instead):
  "ensemble24"    BASELINE config[3]'s advection component, STRONG scaling: 24 BPS-perturbed
                  members x 12 single-step extrapolator calls (nowcasts/utils.py:440-458), members
                  round-robin over the GPUs, motion field estimated on rank 0, ONE NCCL broadcast
                  of it.  At N > 1 the N = 1 shape is also timed (rank 0 alone) -> speed-up.
  "composite4096" BASELINE config[4], STRONG scaling: one 4096^2 composite, LK + 24 leadtimes,
                  output row bands over the GPUs, NCCL all-gather of the motion-field bands.

value  : inputs resident in HBM, device time by CUDA events, L2 flushed between steps.
e2e    : the same step through the public NumPy API with pinned HOST buffers, H2D and
         D2H copies inside the timed region.
roofline: the semi-Lagrangian trajectory kernel (sl_multistep_kernel), algorithmic
         bytes per launch / CUDA-event time of that launch, vs MEASURED_PEAKS.json; a second
         entry rates the same launch against the FP64 pipe (what actually bounds it).
parity : before the line is printed, one step's results are compared with the CPU oracle
         (dense field <= 1e-12 everywhere, extrapolated fields bit-identical); a mismatch raises.
cpu_baseline: the CPU oracle (port of the reference path) on the same workload.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

UNIT = "Mpix/s"

# BASELINE.json configs.  The default (config[1]) is what `metric` is quoted on.
WORKLOADS = {
    "lk_sl12_2048": dict(m=2048, n=2048, T=12, motion="lk", scaling="weak", members=0,
                         metric="Mpix/s advected (2048^2 frame, 12 leadtimes)"),
    "vet_sl12_2048": dict(m=2048, n=2048, T=12, motion="vet", scaling="weak", members=0,
                          metric="Mpix/s advected (2048^2 frame, 12 leadtimes, VET motion)"),
    "composite4096": dict(m=4096, n=4096, T=24, motion="lk", scaling="strong", members=0,
                          metric="Mpix/s advected (4096^2 composite, 24 leadtimes, row bands over GPUs)"),
    # config[3]'s advection component: the call shape of nowcasts/utils.py:441-458 -- every
    # member has its own (perturbed) velocity, precipitation field and carried displacement,
    # one single-step extrapolator call per member and lead time; members sharded over ranks
    "ensemble24": dict(m=2048, n=2048, T=12, motion="lk", scaling="strong", members=24,
                       metric="Mpix/s advected (24-member ensemble, 2048^2, 12 single-step calls per member)"),
}
EXTRAS = ("ensemble24", "composite4096")

# module-level view of the selected headline workload (tests/test_bench_host.py reads these)
M = N_ = 2048
T_LEAD = 12
METRIC = WORKLOADS["lk_sl12_2048"]["metric"]
MOTION = "lk"
SCALING = "weak"
MEMBERS = 0


def set_workload(name):
    global M, N_, T_LEAD, METRIC, MOTION, SCALING, MEMBERS
    w = WORKLOADS[name]
    M, N_, T_LEAD, METRIC, MOTION, SCALING, MEMBERS = (w["m"], w["n"], w["T"], w["metric"], w["motion"],
                                                       w["scaling"], w["members"])
    return dict(w, name=name)


def have_lk():
    try:
        from pysteps_b200.motion import lucaskanade  # noqa: F401
        return True
    except ImportError:
        return False


def workload_name(lk=True, w=None):
    w = w or dict(m=M, n=N_, T=T_LEAD, motion=MOTION, scaling=SCALING, members=MEMBERS)
    mot = {"lk": "lk_dense", "vet": "vet"}[w["motion"]] if lk else "given_field"
    if w["members"]:
        return f"{mot}+semilagrangian_{w['members']}members_x{w['T']}single_steps_{w['m']}x{w['n']}"
    return f"{mot}+semilagrangian_T{w['T']}_{w['m']}x{w['n']}" + ("_rowbands" if w["scaling"] == "strong" else "")


def config_of(w):
    """Identical for both arms (`--impl ours` / `--impl reference`)."""
    return {"workload": workload_name(True, w), "frame": [w["m"], w["n"]], "leadtimes": w["T"]}


def make_inputs(w, seed):
    """frames: float64 (2,m,n) for the motion estimator (as pysteps importers deliver them);
    precip: the last frame as float32 (the synthetic data are float32-exact; a float32 array
    keeps the reference's float64 arithmetic and halves the output volume);
    V: synthetic float32 advection field, used only when the LK stage is not built."""
    from pysteps_b200 import _synthetic as syn
    frames = syn.rain_frames(w["m"], w["n"], 2, seed)
    V = syn.velocity_field(w["m"], w["n"], seed).astype(np.float32)
    return frames, frames[-1].astype(np.float32), V


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock and throttle reasons of rank 0's GPU every 200 ms from the warm-up to the end of the
    timed steps -- the fields of the profiling recipe's nvidia-smi line (clocks.sm, clocks.max.sm,
    the four clocks_event_reasons), read through NVML in a background thread.  An `nvidia-smi -lms`
    loop re-enumerates the box on every poll under a driver-wide lock that kernel launches also take:
    it slowed a launch-heavy step by 40 % on one GPU and by 4x with eight ranks on the box.
    Falls back to the nvidia-smi loop when pynvml is unavailable."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index=0, enabled=True):
        self.index = index
        self.enabled = enabled and not os.environ.get("BENCH_NO_CLOCKS")
        self.samples = []     # (sm_mhz, max_mhz, reason bitmask)
        self.proc = None
        self.thread = None
        self.source = None
        self._stop = False
        self.paused = False   # True inside a timed region: the background thread does not touch NVML there
        self._nv = None

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            import torch
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)

    def _sample(self, nv, h):
        try:
            self.samples.append((nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM),
                                 nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM),
                                 int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))))
        except Exception:
            pass

    def _poll(self, nv, h):
        while not self._stop:
            if not self.paused:
                self._sample(nv, h)
            time.sleep(0.2)

    def sample_now(self):
        """One sample from the CALLING thread.  Used at step boundaries inside the timed region, outside the
        CUDA-event brackets: an NVML query can hold the driver's launch path for tens of ms (one 52 ms step
        in twenty 2.4 ms ones when the background thread's poll fell into the 60 ms timed region); taken
        between two steps it delays nothing that is timed."""
        if self._nv is not None:
            self._sample(*self._nv)

    def __enter__(self):
        if not self.enabled:
            return self
        try:
            import threading
            nv, h = self._nvml_handle()
            self._nv = (nv, h)
            self.source = ("nvml (pynvml): every 200 ms during the warm-up load, at step boundaries inside the "
                           "timed region (outside the event brackets)")
            self.thread = threading.Thread(target=self._poll, args=(nv, h), daemon=True)
            self.thread.start()
            time.sleep(0.25)
            return self
        except Exception:
            self.thread = None
        try:
            self.source = "nvidia-smi -lms 200"
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.25)  # let the first samples arrive before the timed region starts
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *exc):
        if self.thread is not None:
            time.sleep(0.05)
            self._stop = True
            self.thread.join(timeout=2)
        if self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
            except Exception:
                self.proc.kill()
                out = ""
            for line in (out or "").splitlines():
                parts = [x.strip() for x in line.split(",")]
                if len(parts) >= 6 and parts[0].isdigit() and parts[1].isdigit():
                    mask = sum(bit for (nm, bit), v in zip(self.BITS, parts[2:6]) if v.lower() == "active")
                    self.samples.append((int(parts[0]), int(parts[1]), mask))
        if len(self.samples) >= 3:
            self.samples = self.samples[1:]  # the first sample was taken before any load

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(s[0] for s in self.samples)
        reasons = [nm for nm, bit in self.BITS if any(s[2] & bit for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(s[1] for s in self.samples), "reasons": reasons,
                "samples": len(self.samples), "source": self.source}


def stage_rooflines(trace_ms, steps, m, n, peak_gbs, sl_bytes):
    """Per C-ABI call of the step: algorithmic bytes per call (SURVEY.md section 8d figures, with
    the float64 frames this implementation keeps), achieved GB/s over the CUDA-event time of
    the call, fraction of the HBM peak, and what actually bounds it (from the ncu captures in
    profiles/).  `trace_ms` = {name: [ms of every call in the timed region]}."""
    px = m * n
    table = {
        "b200_idw_fill": (16 * px, "alu/latency: exhaustive-in-tile k-NN with register-resident sorted lists"),
        "b200_sl_extrapolate_rows": (sl_bytes, "FP64 pipe + L1 wavefronts + issue (reference-order float64 trajectories)"),
        "b200_min_eig": (5 * px, "latency: one sequential FP64 running sum per column (OpenCV-exact box filter)"),
        "b200_quantise_u8": (10 * px, "hbm/l2 streaming"),
        "b200_mask_invalid": (9 * px, "hbm streaming + reduction"),
        "b200_morph_opening": (17 * px, "hbm/l2 streaming stencil"),
        "b200_masked_minmax": (9 * px, "hbm streaming reduction"),
        "b200_lk_frontend": (26 * px, "hbm streaming (fused mask + min/max, opening + both quantisations)"),
        "b200_lk_track": (None, "latency: ordered float32 window sums, one CTA per feature"),
        "b200_good_features": (None, "latency: sort + ordered greedy selection"),
        "b200_detect_outliers": (None, "latency: cKDTree build (one CTA) + one best-first query per vector"),
        "b200_bps_perturb_velocity": (32 * px, "hbm streaming"),
    }
    out = []
    for name, ms in trace_ms.items():
        if name not in table or not ms:
            continue
        nbytes, bound = table[name]
        avg = sum(ms) / len(ms)
        row = {"call": name, "ms_per_call": avg, "calls_per_step": len(ms) / steps,
               "algorithmic_bytes_per_call": nbytes, "bound": bound}
        if nbytes is not None and avg > 0:
            row["achieved_gbs"] = nbytes / (avg * 1e-3) / 1e9
            row["frac_of_hbm_peak"] = row["achieved_gbs"] / peak_gbs
        out.append(row)
    out.sort(key=lambda r: -r["ms_per_call"] * r["calls_per_step"])
    return out


# ----------------------------------------------------------------------------- CPU legs
_THREADS = {}


def host_threads():
    """Thread count of the CPU legs, set explicitly whatever the launcher exported (torchrun sets
    OMP_NUM_THREADS=1): all logical CPUs, or half of them (one per physical core of an SMT-2
    host) when that runs the oracle's advection kernel faster -- measured once per process."""
    import oracle
    if "n" in _THREADS:
        return oracle.set_num_threads(_THREADS["n"])
    forced = int(os.environ.get("BENCH_CPU_THREADS", "0"))
    ncpu = os.cpu_count() or 1
    if forced or ncpu < 4:
        _THREADS["n"] = forced or ncpu
        return oracle.set_num_threads(_THREADS["n"])
    from oracle import semilagrangian as ora
    from pysteps_b200 import _synthetic as syn
    P, V = syn.rain_field(1024, 1024, 0), syn.velocity_field(1024, 1024, 0)
    best = None
    for cand in (ncpu, ncpu // 2):
        oracle.set_num_threads(cand)
        ora.extrapolate(P, V, 2)
        t0 = time.perf_counter()
        ora.extrapolate(P, V, 4)
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, cand)
    _THREADS["n"] = best[1]
    return oracle.set_num_threads(best[1])


def cpu_step(w, frames, precip, V, lk):
    """The oracle port of one step on host cores; returns seconds of the WHOLE step (ensemble:
    motion + members x the one member that is run).  The k-NN stages run the exhaustive
    lower-index scan (OpenMP C, the faster of the oracle's two modes -- a tougher baseline than
    the reference's single-threaded cKDTree queries)."""
    from oracle import lucaskanade as ora_lk
    from oracle import semilagrangian as ora
    t0 = time.perf_counter()
    if lk and w["motion"] == "vet":
        from oracle import vet as ora_vet
        V = ora_vet.vet(frames, verbose=False)
    elif lk:
        with ora_lk.knn_mode("lower_index"):
            V = ora_lk.dense_lucaskanade(frames)
    if w["members"]:
        # bounded sample: ONE member of the ensemble (the members are independent and identical
        # in cost), extrapolated to all of them
        from oracle import noise_motion as ora_bps
        t1 = time.perf_counter()
        pert = ora_bps.initialize_bps(V, 1.0, 5.0, randstate=np.random.RandomState(1000))
        disp = None
        for t in range(w["T"]):
            Vm = ora_bps.perturbed_velocity(V, pert, (t + 1) * 5.0)
            _, disp = ora.extrapolate(precip, Vm, [1.0], displacement_prev=disp, return_displacement=True)
        member = time.perf_counter() - t1
        return (t1 - t0) + w["members"] * member
    ora.extrapolate(precip, V, w["T"])
    return time.perf_counter() - t0


def cpu_baseline(w, frames, precip, V, lk, reps=2):
    """On the GPU box's host cores: the REFERENCE itself when it travelled (oracle/_ref) on a
    bounded crop (~15 s of CPU work), and the oracle's OpenMP port on the full frame beside it."""
    threads = host_threads()
    times = [cpu_step(w, frames, precip, V, lk) for _ in range(reps)]
    best = min(times)
    port = {"value": (w["members"] or 1) * w["T"] * w["m"] * w["n"] / best / 1e6, "unit": UNIT, "cores": threads,
            "kind": "port",
            "sample": f"{reps} full step(s) of {workload_name(lk, w)} (oracle C/NumPy port, "
                      f"OpenMP {threads} threads, exhaustive k-NN mode), best of {reps}: "
                      + " / ".join(f"{t:.2f}" for t in times) + " s"
                      + (f" (1 of {w['members']} members run, scaled)" if w["members"] else "")}
    if not have_reference():
        return port
    side = 1024 if w["m"] >= 2048 else w["m"] // 2
    r0, c0 = (w["m"] - side) // 2, (w["n"] - side) // 2
    crop = (slice(None), slice(r0, r0 + side), slice(c0, c0 + side))
    t = reference_step(w, np.ascontiguousarray(frames[crop]), np.ascontiguousarray(precip[crop[1:]]),
                       np.ascontiguousarray(V[crop]), lk)
    return {"value": (w["members"] or 1) * w["T"] * side * side / t / 1e6, "unit": UNIT, "cores": threads,
            "kind": "reference",
            "sample": f"1 step of pysteps v1.21.3 itself (oracle/_ref) on a centred {side}x{side} crop of the "
                      f"workload's frames: {t:.1f} s", "port": port}


def reference_step(w, frames, precip, V, lk):
    """One step by the REFERENCE ITSELF (pysteps v1.21.3, unmodified, imported from its compiled form
    oracle/_ref -- or /root/reference where that exists): seconds of the whole step."""
    import contextlib
    import io
    import warnings
    from oracle import refimport
    sl = refimport.ref_module("pysteps.extrapolation.semilagrangian").extrapolate
    with warnings.catch_warnings(), contextlib.redirect_stdout(io.StringIO()):
        warnings.simplefilter("ignore")
        t0 = time.perf_counter()
        if lk and w["motion"] == "vet":
            V = refimport.ref_module("pysteps.motion.vet").vet(frames, verbose=False)
        elif lk:
            V = refimport.ref_module("pysteps.motion.lucaskanade").dense_lucaskanade(frames)
        if w["members"]:
            bps = refimport.ref_module("pysteps.noise.motion")
            t1 = time.perf_counter()
            pert = bps.initialize_bps(V, 1.0, 5.0, randstate=np.random.RandomState(1000))
            disp = None
            for t in range(w["T"]):
                Vm = V + bps.generate_bps(pert, (t + 1) * 5.0)
                _, disp = sl(precip, Vm, [1.0], displacement_prev=disp, return_displacement=True)
            member = time.perf_counter() - t1
            return (t1 - t0) + w["members"] * member
        sl(precip, V, w["T"])
        return time.perf_counter() - t0


def have_reference():
    try:
        from oracle import refimport
        return refimport.available(extensions=True)
    except Exception:
        return False


def run_reference(args, w):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    lk = have_lk_oracle()
    frames, precip, V = make_inputs(w, 0)
    threads = host_threads()
    real = have_reference() and not os.environ.get("BENCH_REFERENCE_PORT_ONLY")
    step = reference_step if real else cpu_step
    kind = "reference" if real else "port"
    what = ("pysteps v1.21.3 itself (oracle/_ref: its modules as bytecode + its Cython extensions built with "
            "setup.py's flags), stock dense_lucaskanade / extrapolate: SciPy cKDTree and map_coordinates are "
            "single-threaded by construction, OpenCV and the extensions use the host's threads") if real else \
        f"oracle port of the reference path, OpenMP {threads} threads (set explicitly), exhaustive k-NN mode"
    small = (slice(None), slice(0, 256), slice(0, 256))
    for _ in range(args.warmup):
        step(w, np.ascontiguousarray(frames[small]), np.ascontiguousarray(precip[small[1:]]),
             np.ascontiguousarray(V[small]), lk)
    # Every step is a bounded sample of the workload: the full frame when the host is fast enough
    # for the whole run to end within a few minutes, else a centred crop sized from the first
    # step's time (stated in `sample`); the metric is per advected pixel.
    budget_s = float(os.environ.get("BENCH_REFERENCE_BUDGET_S", "240"))
    dt = step(w, frames, precip, V, lk)
    first = dt
    m, n = w["m"], w["n"]
    pixels = m * n
    sample = f"every step on the full {m}x{n} frame"
    side_m, side_n = m, n
    fr_c, pr_c, V_c = frames, precip, V
    if dt * args.steps > budget_s and args.steps > 1:
        frac = max((budget_s - dt) / (dt * (args.steps - 1)), 1.0 / 64.0)
        side_m = max(256, int(m * frac ** 0.5) // 32 * 32)
        side_n = max(256, int(n * frac ** 0.5) // 32 * 32)
        r0, c0 = (m - side_m) // 2, (n - side_n) // 2
        fr_c = np.ascontiguousarray(frames[:, r0:r0 + side_m, c0:c0 + side_n])
        pr_c = np.ascontiguousarray(precip[r0:r0 + side_m, c0:c0 + side_n])
        V_c = np.ascontiguousarray(V[:, r0:r0 + side_m, c0:c0 + side_n])
        sample = (f"first step on the full frame ({dt:.1f} s), the other {args.steps - 1} on a centred "
                  f"{side_m}x{side_n} crop to stay within {budget_s:.0f} s")
    for _ in range(args.steps - 1):
        dt += step(w, fr_c, pr_c, V_c, lk)
        pixels += side_m * side_n
    val = (w["members"] or 1) * w["T"] * pixels / dt / 1e6
    line = {"impl": "reference", "metric": w["metric"], "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": w["scaling"], "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": config_of(w),
            "note": "host throughput: N independent nowcasts take N times as long on the same cores, so the "
                    "Mpix/s of this arm is the same at every --gpus N",
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": kind,
                             "sample": f"{args.steps} step(s), {sample}; {what}"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if real:
        # the tougher figure beside it: the oracle's OpenMP C/NumPy port of the same path, one full step
        tp = cpu_step(w, frames, precip, V, lk)
        line["port"] = {"value": (w["members"] or 1) * w["T"] * m * n / tp / 1e6, "unit": UNIT, "cores": threads,
                        "kind": "port", "sample": f"1 full step, {tp:.2f} s (first reference step: {first:.1f} s)"}
    print(json.dumps(line))
    return 0


def have_lk_oracle():
    try:
        from oracle import lucaskanade  # noqa: F401
        return have_lk()
    except ImportError:
        return False


# ----------------------------------------------------------------------------- GPU arm
def settle_gc():
    """Before a timed region: collect, then move everything alive to CPython's permanent generation
    (gc.freeze).  A generation-2 collection of a process that has imported torch walks millions of objects
    -- 50-60 ms, more than twenty 2.4 ms steps -- and fires wherever the allocation counter happens to
    trip, e.g. inside a torch.empty of step 13.  It is a property of the interpreter's heap, not of the
    path measured here; every line says `gc: frozen` so that the choice is visible."""
    gc.collect()
    gc.freeze()


class Bench:
    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        import pysteps_b200
        from pysteps_b200 import _lib, _shard
        self.pkg, self.lib, self.shard = pysteps_b200, _lib, _shard
        self.extrap = pysteps_b200.extrapolation.get_method("semilagrangian")
        self.lk = have_lk()
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB L2
        self.last_out = None

    def motion(self, name):
        if not self.lk:
            return None
        f = self.pkg.motion.get_method(name)
        if name == "vet":
            torch = self.torch
            return lambda fr, **kw: f(fr.cpu().numpy() if torch.is_tensor(fr) else fr, verbose=False)
        return f

    def pin(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def all_agree(self, flag):
        """rank 0 decides, so every rank runs the same number of steps"""
        if self.world == 1:
            return bool(flag)
        t = self.torch.tensor([int(flag)], device="cuda")
        self.dist.broadcast(t, src=0)
        return bool(t.item())

    def time_device(self, step, steps, warmup, min_warm_s=0.0, marks=None, sampler=None, keep_last=False):
        """W >= 3 untimed steps (stretched to min_warm_s of the same load for the clock sampler),
        then `steps` steps, each bracketed by barrier + synchronize and CUDA events, L2 flushed in
        between (outside the events).  Returns (ms summed over steps [max over ranks], trace,
        launches, per-phase ms when the step records `marks`).  keep_last: the last timed step's
        result is left in self.last_out (earlier results are dropped as they come, so the allocator
        sees the same pattern as without it)."""
        torch = self.torch
        t_w, n_w = time.perf_counter(), 0
        while True:
            step()
            torch.cuda.synchronize()
            n_w += 1
            if self.all_agree(n_w >= warmup and (n_w >= 400 or time.perf_counter() - t_w >= min_warm_s)):
                break
        self.barrier()
        settle_gc()
        step()  # one more untimed step: whatever the collection left to be re-established is paid here
        torch.cuda.synchronize()
        self.barrier()
        launches0 = self.lib.load().b200_launch_count()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        phase = []
        # inside the timed region only the rated kernel's call carries CUDA events (two events per
        # traced call cost ~15 us of host time: 14 ms of an ensemble step when every call is traced)
        if sampler is not None:
            sampler.paused = True
        with self.lib.Trace(only=("b200_sl_extrapolate_rows", "b200_sl_extrapolate")) as trace:
            for i, (s, e) in enumerate(ev):
                if sampler is not None and i in (1, steps // 2, steps - 1):
                    sampler.sample_now()  # the previous step is still executing: a sample under load
                self.flush.fill_(1)
                self.barrier()
                s.record()
                if keep_last and i == steps - 1:
                    self.last_out = step()
                else:
                    step()
                e.record()
                if marks is not None:
                    phase.append(list(marks))
            if sampler is not None:
                sampler.sample_now()
            self.barrier()
        if sampler is not None:
            sampler.paused = False
        launches = self.lib.load().b200_launch_count() - launches0
        self.each_ms = [s.elapsed_time(e) for s, e in ev]  # this rank's steps, one by one
        dev_ms = self.shard.max_over_ranks(sum(self.each_ms), device="cuda")
        # per-stage table: two more, untimed, fully traced steps
        with self.lib.Trace() as stage_trace:
            for _ in range(2):
                self.flush.fill_(1)
                self.barrier()
                step()
            self.barrier()
        self.stage_trace = {k: v for k, v in stage_trace.summary().items()}
        self.stage_steps = 2
        phases = None
        if marks is not None and phase and len(phase[0]) >= 1:
            # phase boundaries recorded by the step (events on the current stream)
            acc = [0.0] * (len(phase[0]) + 1)
            for (s, e), mk in zip(ev, phase):
                pts = [s] + mk + [e]
                for i in range(len(pts) - 1):
                    acc[i] += pts[i].elapsed_time(pts[i + 1])
            phases = [self.shard.max_over_ranks(a, device="cuda") / steps for a in acc]
        return dev_ms, trace.summary(), launches, phases

    def time_host(self, step, steps, warmup):
        # the pinned host pool (torch's caching host allocator: one cudaHostAlloc per new block, tens
        # of ms for a 200 MB result) reaches its steady state after a few calls
        out = None
        for _ in range(max(4, warmup)):
            out = step()
        self.barrier()
        settle_gc()
        t0 = time.perf_counter()
        for _ in range(steps):
            out = step()
        self.barrier()
        return self.shard.max_over_ranks(time.perf_counter() - t0, device="cuda"), out


def build_standard(b, w, active=None):
    """config[1] / [2] / [4]: motion field + T-leadtime extrapolation.  Returns step functions and
    byte counts; `active` = ranks taking part (None: all)."""
    torch, dist, world, rank = b.torch, b.dist, b.world, b.rank
    m, n, T = w["m"], w["n"], w["T"]
    frames_h, precip_h, V_h = (b.pin(a) for a in make_inputs(w, rank))
    frames_d = torch.from_numpy(frames_h).cuda()
    precip_d = torch.from_numpy(precip_h).cuda()
    V_d = torch.from_numpy(V_h).cuda()
    motion = b.motion(w["motion"])
    lk = motion is not None
    strong = w["scaling"] == "strong"
    band = b.shard.row_band(m, world, rank) if strong else None
    ekw = {} if band is None else {"b200_rows": band}
    extrap = b.extrap

    def step_device():
        if lk and strong and world > 1 and w["motion"] == "lk":
            # one composite over GPUs: the sparse LK stages are deterministic and replicated, every
            # rank fills its band of the motion field, the bands are all-gathered (the exchange
            # step of this path), and every rank advects its band of output rows
            Vband = motion(frames_d, interp_kwargs={"b200_rows": band})
            Vd = b.shard.gather_row_bands(Vband, m, world, rank)
            return extrap(precip_d, Vd, T, **ekw)
        if lk:
            Vd = motion(frames_d)
            if not torch.is_tensor(Vd):
                Vd = torch.from_numpy(np.ascontiguousarray(Vd)).cuda()
            return extrap(precip_d, Vd, T, **ekw)
        return extrap(precip_d, V_d, T, **ekw)

    def step_host():
        """public NumPy API: H2D of inputs and D2H of the result inside."""
        if lk and strong and world > 1 and w["motion"] == "lk":
            # host frames in, host result out; the motion-field bands meet on the devices (NCCL)
            Vband = motion(torch.from_numpy(frames_h).cuda(non_blocking=True), interp_kwargs={"b200_rows": band})
            Vh = b.shard.gather_row_bands(Vband, m, world, rank)
        elif lk:
            Vh = motion(frames_h)  # NumPy (2,m,n) float64, as pysteps returns it
        else:
            Vh = V_h
        return extrap(precip_h, Vh, T, **ekw)

    rows_here = m if band is None else band[1] - band[0]
    # LK: frames up, field down, field up again for the extrapolator (the plugin API is NumPy;
    # the second upload is served from the device copy the motion call left behind, see
    # pysteps_b200/_device.py: recent_results)
    h2d = precip_h.nbytes + (frames_h.nbytes if lk else V_h.nbytes)
    d2h = rows_here * n * 4 * T + (2 * m * n * 8 if (lk and not (strong and world > 1)) else 0)
    info = dict(h2d=h2d, d2h=d2h, rows_here=rows_here, lk=lk, inputs=(frames_h, precip_h, V_h),
                dev_inputs=(frames_d, precip_d, V_d), nfields=(world if w["scaling"] == "weak" else 1))
    return step_device, step_host, info


def build_ensemble(b, w, solo=False):
    """config[3]'s advection component.  solo=True: the N = 1 shape inside an N > 1 job (rank 0
    runs all members, the other ranks idle) -- the denominator of the speed-up."""
    torch, dist, world, rank = b.torch, b.dist, b.world, b.rank
    m, n, T, members = w["m"], w["n"], w["T"], w["members"]
    frames_h, precip_h, _ = (b.pin(a) for a in make_inputs(w, 0))
    frames_d = torch.from_numpy(frames_h).cuda()
    precip_d = torch.from_numpy(precip_h).cuda()
    motion = b.motion("lk")
    bps_init, bps_gen = b.pkg.noise.get_method("bps")
    eff_world = 1 if solo else world
    mine = b.shard.member_indices(members, eff_world, rank) if (not solo or rank == 0) else []
    # per-member precipitation fields (synthetic); the velocity perturbations are the BPS
    # perturbator's (noise/motion.py), one seeded RandomState per member as in
    # nowcasts/steps.py:915-926, evaluated inside the advection call (fused kernel)
    member_precip = [precip_d * (1.0 + 0.01 * i) for i in mine]
    member_precip_h = [b.pin(precip_h * np.float32(1.0 + 0.01 * i)) for i in mine]
    KMPP, DT_MIN = 1.0, 5.0
    extrap = b.extrap
    marks = []

    def member_loop(V, fields, resident):
        """nowcasts/utils.py:440-458: T lead times x this rank's members, each a single-step
        call with a freshly perturbed motion field, carrying its own displacement."""
        perts = [bps_init(V, 1.0 / KMPP, DT_MIN, randstate=np.random.RandomState(1000 + i)) for i in mine]
        disp = [None] * len(mine)
        last = None
        for t in range(T):
            for j in range(len(mine)):
                Vm = V + bps_gen(perts[j], (t + 1) * DT_MIN)
                last, disp[j] = extrap(fields[j], Vm, [1.0], displacement_prev=disp[j],
                                       return_displacement=True, b200_resident=resident)
        return last

    from pysteps_b200.extrapolation.semilagrangian import extrapolate_members
    stack = torch.stack(member_precip) if member_precip else None

    def member_loop_batched(V):
        """the same member-steps through the batched entry point: all members of this rank in one
        perturbation launch + one trajectory launch per lead time (b200_sl_step_batched)"""
        perts = [bps_init(V, 1.0 / KMPP, DT_MIN, randstate=np.random.RandomState(1000 + i)) for i in mine]
        disp, last = None, None
        for t in range(T):
            Vm = [V + bps_gen(pt, (t + 1) * DT_MIN) for pt in perts]
            last, disp = extrapolate_members(stack, Vm, displacement_prev=disp)
        return last

    def step_device_batched():
        if solo and rank != 0:
            return None
        if rank == 0:
            Vd = motion(frames_d)
        else:
            Vd = torch.empty((2, m, n), dtype=torch.float64, device="cuda")
        if not solo:
            Vd = b.shard.broadcast_field(Vd, src=0)
        return member_loop_batched(Vd) if mine else None

    def step_device():
        """rank 0: motion field; broadcast; member loop on device-resident fields."""
        del marks[:]
        if solo and rank != 0:  # idle rank of the N = 1 shape: same phase marks, no work
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            marks.append(ev)
            return None
        if rank == 0:
            Vd = motion(frames_d)
        else:
            Vd = torch.empty((2, m, n), dtype=torch.float64, device="cuda")
        if not solo:
            Vd = b.shard.broadcast_field(Vd, src=0)  # the only collective (NCCL over NVLink)
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        marks.append(ev)
        return member_loop(Vd, member_precip, False)

    def step_host():
        # NumPy API as nowcast_main_loop uses it: the motion field is uploaded once per
        # forecast, every member-step uploads its precipitation field and downloads the
        # advected one; perturbed fields and displacements never leave the device
        if solo and rank != 0:
            return None
        Vh = motion(frames_h) if rank == 0 else None
        if world > 1 and not solo:
            Vd = torch.from_numpy(Vh).cuda() if rank == 0 else \
                torch.empty((2, m, n), dtype=torch.float64, device="cuda")
            dist.broadcast(Vd, src=0)
            Vh = Vd.cpu().numpy()
        return member_loop(Vh, member_precip_h, True)

    # per rank: frames + field once, one precipitation field up / one down per member-step
    h2d = frames_h.nbytes + 2 * m * n * 8 + len(mine) * T * precip_h.nbytes
    d2h = 2 * m * n * 8 + len(mine) * T * precip_h.nbytes
    info = dict(h2d=h2d, d2h=d2h, rows_here=m, lk=True, nfields=members, marks=marks, members_here=len(mine),
                step_device_batched=step_device_batched)
    return step_device, step_host, info


def parity_check(b, w):
    """One step of the headline workload, CUDA vs the CPU oracle on the same inputs (rank 0's):
    dense motion field <= 1e-12 at every pixel against the oracle in the reference's k-NN order,
    sparse vectors and the T extrapolated fields bit-identical.  Raises on a mismatch."""
    torch = b.torch
    from oracle import lucaskanade as ora_lk
    from oracle import semilagrangian as ora_sl
    t0 = time.perf_counter()
    frames, precip, Vsyn = make_inputs(w, 0)
    res = {"checked": workload_name(True, w)}
    V = Vsyn
    if b.lk and w["motion"] == "lk":
        lk = b.motion("lk")
        xy, uv = lk(frames, dense=False)
        oxy, ouv = ora_lk.dense_lucaskanade(frames, dense=False)
        if not (np.array_equal(xy, oxy) and np.array_equal(uv, ouv)):
            raise AssertionError("bench parity: sparse Lucas-Kanade vectors differ from the oracle")
        V = lk(frames)
        Vo = ora_lk.dense_lucaskanade(frames)
        d = float(np.abs(V - Vo).max())
        res.update(sparse_vectors=int(len(xy)), sparse_bit_identical=True, dense_field_max_abs_diff=d,
                   dense_field_tolerance=1e-12)
        if not d <= 1e-12:
            raise AssertionError(f"bench parity: dense motion field differs from the oracle by {d:.3e}")
    got = b.extrap(precip, V, w["T"])
    want = ora_sl.extrapolate(precip, V, w["T"])
    same = np.array_equal(np.isnan(got), np.isnan(want)) and np.array_equal(got[~np.isnan(got)], want[~np.isnan(want)])
    res.update(extrapolation_bit_identical=bool(same), seconds=round(time.perf_counter() - t0, 1))
    if not same:
        raise AssertionError("bench parity: extrapolated fields are not bit-identical to the oracle")
    return res


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


# FP64 pipe of sm_100a: 64 results per SM per clock (B200: 40 TFLOP/s FP64 FMA = 20e12 instr/s over
# 148 SMs at 1.965 GHz -> 68.8, i.e. 64/clk); instruction count per pixel-leadtime of
# sl_multistep_kernel from its SASS (tools/sass_count.py, profiles/r02_sl_kernel.md)
FP64_PER_CLK_SM = 64
SL_FP64_INSTR_PER_PIXEL_LEADTIME = 94


DUMP_LIMIT = 64 * 10 ** 6  # bytes written by --dump-outputs, all files together
# what --dump-outputs writes for a pixel the extrapolation leaves undefined (outval=nan: advected in from
# outside the domain).  The dumped fields are precipitation (>= 0), so the value cannot be a real one.
DUMP_UNDEFINED = -9999.0


def dump_outputs(out, dirpath):
    """Writes what one step of the timed path returned as DIR/<name>.npy (float32 / float64).  An
    array larger than its share of DUMP_LIMIT is cut to a fixed, seeded sample of rows (axis -2),
    the same rows on every run, so that two builds can be compared output for output.  The files hold
    finite numbers only: NaN is written as DUMP_UNDEFINED, which a dumped field never holds otherwise
    (checked here, as is the absence of infinities)."""
    arrays = list(out) if isinstance(out, (tuple, list)) else [out]
    names = ["extrapolated"] if len(arrays) == 1 else [f"extrapolated_{i}" for i in range(len(arrays))]
    budget = DUMP_LIMIT // len(arrays) - 4096  # room for the .npy header
    os.makedirs(dirpath, exist_ok=True)
    written = {}
    for name, a in zip(names, arrays):
        a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float64)
        shape = list(a.shape)
        if a.nbytes > budget:
            rows = a.shape[-2]
            keep = max(1, budget * rows // a.nbytes)
            a = a[..., np.sort(np.random.default_rng(0).choice(rows, keep, replace=False)), :]
        nan = np.isnan(a)
        if np.isinf(a).any() or (a == DUMP_UNDEFINED).any():
            raise ValueError(f"--dump-outputs: {name} holds an infinity or the value {DUMP_UNDEFINED}")
        np.save(os.path.join(dirpath, name + ".npy"), np.ascontiguousarray(np.where(nan, a.dtype.type(DUMP_UNDEFINED), a)))
        written[name] = {"shape": shape, "saved_shape": list(a.shape), "dtype": str(a.dtype),
                         "undefined_written_as": DUMP_UNDEFINED, "undefined": int(np.count_nonzero(nan))}
    return written


def measure(b, w, steps, warmup, clocks=None, solo=False, dump=None):
    """device-resident + end-to-end timing of one workload -> dict (rank 0) / None.  dump: directory
    that receives the last timed step's result (dump_outputs)."""
    if w["members"]:
        step_device, step_host, info = build_ensemble(b, w, solo=solo)
    else:
        step_device, step_host, info = build_standard(b, w)
    m, n, T = w["m"], w["n"], w["T"]
    marks = info.get("marks")
    if clocks is not None:
        clocks.__enter__()
    dev_ms, tr, launches, phases = b.time_device(step_device, steps, warmup, 0.5 if clocks is not None else 0.0, marks,
                                                 sampler=clocks, keep_last=dump is not None)
    each_ms = list(b.each_ms)
    if clocks is not None:
        clocks.__exit__(None, None, None)
    dumped = None
    if dump is not None:
        if b.rank == 0 and b.last_out is not None:
            dumped = dump_outputs(b.last_out, dump)
        b.last_out = None
    nfields = info["nfields"]
    value = nfields * steps * T * m * n / (dev_ms * 1e-3) / 1e6
    stage_trace, stage_steps = b.stage_trace, b.stage_steps
    ms_b = None
    if w["members"] and not solo:
        # the same ensemble step with the members of a rank batched into one launch per lead time
        ms_b, _, _, _ = b.time_device(info["step_device_batched"], steps, warmup)
    e2e_s, out = b.time_host(step_host, steps, warmup)
    e2e_val = nfields * steps * T * m * n / e2e_s / 1e6
    if b.rank != 0:
        return None
    world = 1 if solo else b.world
    blk = {"metric": w["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
           "ms_per_step": dev_ms / steps, "higher_is_better": True, "scaling": w["scaling"],
           "config": config_of(w),
           "parallelism": (
               f"{world} independent nowcast(s), one per GPU, no collective" if w["scaling"] == "weak" else
               f"{w['members']} members round-robin over {world} GPU(s), NCCL broadcast of the motion field"
               if w["members"] else
               f"output row bands over {world} GPU(s), inputs replicated"
               + (", NCCL all-gather of the motion-field bands" if world > 1 and w["motion"] == "lk" else "")),
           "fields_per_gpu": 1 if w["scaling"] == "weak" else round(1.0 / world, 4),
           "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(info["h2d"]),
                   "d2h_bytes_per_step": int(info["d2h"]), "ms_per_step": 1e3 * e2e_s / steps},
           "gpu_launches": int(launches), "ms_each_step_rank0": [round(x, 3) for x in each_ms], "gc": "frozen",
           "_trace": tr, "_info": info,
           "_stage_trace": stage_trace, "_stage_steps": stage_steps}
    if phases is not None and len(phases) == 2:
        blk["motion_and_broadcast_ms"] = phases[0]
        blk["member_loop_ms"] = phases[1]
    if ms_b is not None:
        blk["batched_ms_per_step"] = ms_b / steps
        blk["batched_value"] = nfields * steps * T * m * n / (ms_b * 1e-3) / 1e6
        blk["batched_note"] = ("extrapolate_members / b200_sl_step_batched (all members of a rank in one launch "
                               "per lead time): not a call the unmodified nowcast_main_loop makes; `value` is "
                               "the per-member call shape")
    if dumped is not None:
        blk["dumped_outputs"] = dumped
    return blk


def roofline_of(b, w, blk, peaks):
    tr, info = blk["_trace"], blk["_info"]
    m, n, T = w["m"], w["n"], w["T"]
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650"
    k_ms = tr.get("b200_sl_extrapolate_rows", []) or tr.get("b200_sl_extrapolate", [])
    k_avg = sum(k_ms) / len(k_ms) if k_ms else float("nan")
    vbytes = 8 if info["lk"] else 4  # LK returns float64 fields, synthetic V is float32
    alg_bytes = m * n * (2 * vbytes + 4) + info["rows_here"] * n * 4 * T
    pix_leadtimes = info["rows_here"] * n * T
    if w["members"]:  # single-step member calls: V 16 + precip 4 + displacement in/out 32 + out 4 B per pixel
        alg_bytes = m * n * 56
        pix_leadtimes = m * n
    achieved = alg_bytes / (k_avg * 1e-3) / 1e9
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "sl_traffic.json")))["bytes_per_launch"]
    except Exception:
        pass
    sm_mhz = float(peaks.get("sm_max_mhz", 1965.0))
    nsm = b.torch.cuda.get_device_properties(0).multi_processor_count
    fp64_peak = FP64_PER_CLK_SM * nsm * sm_mhz * 1e6 / 1e9  # G instr/s
    fp64_ach = SL_FP64_INSTR_PER_PIXEL_LEADTIME * pix_leadtimes * (2 if w["members"] else 1) / (k_avg * 1e-3) / 1e9
    roofline = {"kernel": "sl_multistep_kernel", "bound": "hbm", "achieved": achieved,
                "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "peak_source": peak_src, "kernel_ms": k_avg, "algorithmic_bytes_per_launch": alg_bytes}
    roofline_fp64 = {"kernel": "sl_multistep_kernel", "bound": "fp64 pipe (what limits this kernel: the reference's "
                     "float64 operation order is kept, ~%d FP64 instructions and 36 gathered taps per pixel-leadtime "
                     "against 5 B of compulsory traffic)" % SL_FP64_INSTR_PER_PIXEL_LEADTIME,
                     "achieved": fp64_ach, "peak": fp64_peak, "unit": "G FP64 instr/s", "frac": fp64_ach / fp64_peak,
                     "peak_source": f"{FP64_PER_CLK_SM} FP64 results/clk/SM x {nsm} SMs x {sm_mhz:.0f} MHz",
                     "kernel_ms": k_avg}
    return roofline, roofline_fp64, peak, alg_bytes


def float32_taps_block(b, w, peaks, reps=10):
    """The OPT-IN float32-tap trajectory kernel timed beside the exact one on this workload's motion field
    (device-resident inputs, L2 flushed, CUDA events around each C call).  Its call contains the float64 ->
    float32 copy of the field and the exact fix-up launch over the uncertified pixels, so `ms_per_call` is
    what a user pays; the exact path's `interleave` call is listed beside its kernel for the same reason."""
    import pysteps_b200
    from pysteps_b200 import _lib
    torch = b.torch
    m, n, T = w["m"], w["n"], w["T"]
    frames, precip, _ = make_inputs(w, 0)
    P = torch.from_numpy(precip).cuda()
    V = pysteps_b200.motion.get_method("lk")(torch.from_numpy(frames).cuda())
    extrap = pysteps_b200.extrapolation.get_method("semilagrangian")

    def timed(names, **kw):
        for _ in range(3):
            extrap(P, V, T, **kw)
        acc = {k: [] for k in names}
        for _ in range(reps):
            b.flush.fill_(1)
            with _lib.Trace(only=names) as tr:
                extrap(P, V, T, **kw)
            for k, v in tr.summary().items():
                acc[k] += v
        return {k: sum(v) / len(v) for k, v in acc.items() if v}

    ex = timed(("b200_sl_extrapolate_rows", "b200_sl_interleave_velocity"))
    fa = timed(("b200_sl_extrapolate_rows_f32", "b200_sl_interleave_velocity"), b200_float32_taps=True)
    exact, dex = extrap(P, V, T, return_displacement=True)
    cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
    fast, dfa = extrap(P, V, T, return_displacement=True, b200_float32_taps=True, b200_fallback_count=cnt)
    err = torch.nan_to_num((fast.double() - exact.double()).abs(), nan=0.0).max().item()
    gy, gx = torch.meshgrid(torch.arange(m, device="cuda", dtype=torch.float64),
                            torch.arange(n, device="cuda", dtype=torch.float64), indexing="ij")
    same_idx = bool(torch.equal(torch.floor(gx + dfa[0]), torch.floor(gx + dex[0]))
                    and torch.equal(torch.floor(gy + dfa[1]), torch.floor(gy + dex[1])))
    peak = float(peaks.get("hbm_gbs", 6650.0))
    alg = m * n * (8 + 4 + 4 * T)  # float32 field pairs + float32 precip in + T float32 planes out
    call_ms = fa["b200_sl_extrapolate_rows_f32"]
    return {"what": "opt-in b200_float32_taps=True: float32 taps, float64 trajectory, tap indices certified equal to "
                    "the exact kernel's, uncertified pixels recomputed by the exact code (csrc/sl.cu sl_f32_kernel)",
            "ms_per_call": call_ms, "interleave_ms": fa.get("b200_sl_interleave_velocity"),
            "exact_ms_per_call": ex["b200_sl_extrapolate_rows"], "exact_interleave_ms": ex.get("b200_sl_interleave_velocity"),
            "speedup_vs_exact_call": ex["b200_sl_extrapolate_rows"] / call_ms,
            "recomputed_fraction": cnt.item() / (m * n),
            "max_value_error_over_max_precip": err / float(P.abs().max()),
            "max_displacement_error_px": (dfa - dex).abs().max().item(),
            "tap_indices_equal": same_idx,
            "nan_pattern_equal": bool(torch.equal(torch.isnan(fast), torch.isnan(exact))),
            "roofline": {"bound": "hbm", "achieved": alg / (call_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg / (call_ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": alg}}


def public(blk):
    return {k: v for k, v in blk.items() if not k.startswith("_")}


def run_ours(args, w):
    b = Bench()
    peaks = load_peaks()
    clocks = ClockSampler(b.local, enabled=(b.rank == 0))
    head = measure(b, w, args.steps, args.warmup, clocks=clocks, dump=args.dump_outputs)
    extras = {}
    if not args.no_extras and args.workload == "lk_sl12_2048":
        for name in EXTRAS:
            we = dict(WORKLOADS[name], name=name)
            es = max(3, min(args.steps, args.extra_steps))
            blk = measure(b, we, es, 3)
            solo = None
            if b.world > 1 and we["members"]:
                solo = measure(b, we, 2, 3, solo=True)
            if b.rank == 0:
                if solo is not None:
                    blk["one_gpu_ms_per_step"] = solo["ms_per_step"]
                    blk["speedup_vs_1gpu"] = solo["ms_per_step"] / blk["ms_per_step"]
                    if "member_loop_ms" in solo and "member_loop_ms" in blk:
                        blk["one_gpu_member_loop_ms"] = solo["member_loop_ms"]
                        blk["advection_speedup_vs_1gpu"] = solo["member_loop_ms"] / blk["member_loop_ms"]
                    blk["one_gpu_e2e_ms_per_step"] = solo["e2e"]["ms_per_step"]
                    blk["e2e_speedup_vs_1gpu"] = solo["e2e"]["ms_per_step"] / blk["e2e"]["ms_per_step"]
                r, r64, _, _ = roofline_of(b, we, blk, peaks)
                blk["roofline"] = r
                extras[name] = public(blk)
    if b.rank == 0:
        roofline, roofline_fp64, peak, alg_bytes = roofline_of(b, w, head, peaks)
        tr = head["_stage_trace"]
        stage_ms = {k: sum(v) / head["_stage_steps"] for k, v in tr.items()}
        try:
            stages = stage_rooflines(tr, head["_stage_steps"], w["m"], w["n"], peak, alg_bytes)
        except Exception as exc:  # supplementary table only
            stages = [{"error": repr(exc)}]
        parity = None if args.no_parity else parity_check(b, w)
        # the CPU leg is a property of the host, measured once: rank 0 of the single-GPU run only
        fr, pr, Vh = head["_info"]["inputs"] if "inputs" in head["_info"] else make_inputs(w, 0)
        cpu = cpu_baseline(w, np.asarray(fr), np.asarray(pr), np.asarray(Vh), have_lk_oracle()) \
            if (not args.no_cpu and b.world == 1) else None
        line = public(head)
        line.update({"vs_baseline": None,
                     "dtype": "f64 (trajectories, motion field, IDW); f32 precip in/out; u8/i16/f32 "
                              "OpenCV-exact LK stages", "data": "synthetic",
                     "l2": "flushed between timed steps (256 MB fill)",
                     "clocks": clocks.summary(), "roofline": roofline, "roofline_fp64": roofline_fp64,
                     "parity": parity, "cpu_baseline": cpu, "stage_ms_per_step": stage_ms,
                     "stage_rooflines": stages})
        line.update(extras)
        if not args.no_extras and args.workload == "lk_sl12_2048" and b.world == 1 and b.lk:
            try:
                line["sl_float32_taps"] = float32_taps_block(b, w, peaks)
            except Exception as exc:  # supplementary block only
                line["sl_float32_taps"] = {"error": repr(exc)}
        print(json.dumps(line))
    else:
        if not args.no_parity:
            pass  # rank 0 checks; the others wait at the final barrier
    b.barrier()
    if b.world > 1:
        b.dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of one step")
    ap.add_argument("--no-extras", action="store_true", help="headline workload only")
    ap.add_argument("--extra-steps", type=int, default=5, help="timed steps of the ensemble24 / composite4096 blocks")
    ap.add_argument("--workload", default="lk_sl12_2048", choices=sorted(WORKLOADS))
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline's last timed step's result to DIR/<name>.npy, NaN as -9999 "
                         "(at most 64 MB, a fixed seeded sample of rows beyond that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    w = set_workload(args.workload)
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args, w)
    return run_ours(args, w)


if __name__ == "__main__":
    sys.exit(main())
