#!/usr/bin/env python
"""bench.py -- decoded syndromes/s of batchdecode! on the B200 path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C3] [--per P] [--batch B]
  python bench.py --impl reference ...      # the CPU restatement of the reference, all host threads
  python bench.py --single-process --gpus N # ONE decoder over devices 0..N-1, one 10M-syndrome host batch (strong scaling)

One "step" = one batchdecode! of the whole synthetic batch (default: config C3 of BASELINE.json,
the [[144,12,12]] gross code, 10M syndromes per GPU, max_iters = 32, reference early-stop
semantics).  `value` is measured with the packed syndromes already resident in HBM, `e2e` through
the C-ABI host-buffer call (host BitMatrix in, BitMatrix + success out, copies inside the timed
region; `e2e_by_format` adds pageable buffers and the Matrix{Int} input of the reference's own test).
Under torchrun every rank decodes its own 10M-syndrome shard (weak scaling, inputs keyed by the
global syndrome index) and the counters are all-reduced over NCCL.  At N = 1 a second JSON line, on
stderr, carries extra operating points and short sub-records of the other BASELINE configs at their
full batch sizes (C2 per sweep, C4 10M tiled, C5 1M streamed).

  python bench.py --dump-outputs DIR ...    # also write what the last timed step computed to DIR/*.npy
"""
import argparse
import glob
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402

SEED_E = 12345
METRIC = "decoded syndromes/sec (batchdecode!)"
UNIT = "syndromes/s"
# FP64-pipe issue slots per edge-iteration (DESIGN.md "Rooflines").
#   exact : the reference arithmetic is 10 add/sub/mul + 2 IEEE divisions of D = 8 FP64-pipe instructions each = 26
#           (the algorithmic model of SURVEY 8(d)); the kernels EXECUTE 21 (products with +-1 and unread values dropped).
#   minsum: 2 compares + 1 multiply per edge on the check side, 2 additions on the variable side = 5; no divisions.
FP64_SLOTS = {"exact": {"model": 26, "executed": 21}, "minsum": {"model": 5, "executed": 5}, "fast": {"model": 4, "executed": 4}}
FP64_LANES_PER_SM_CLK = 64
WORKLOAD_NAMES = {"C1": "Gallager (1000,10,9)", "C2": "d=15 rotated surface X checks", "C3": "[[144,12,12]] gross code H_X",
                  "C4": "HGP of Gallager(32,4,3) H_X", "C5": "Gallager (100002,6,3)"}
DEFAULT_PER = {"C1": 0.01, "C2": 0.01, "C3": 0.03, "C4": 0.02, "C5": 0.02}
DEFAULT_B = {"C1": 4096, "C2": 1_000_000, "C3": 10_000_000, "C4": 10_000_000, "C5": 1_000_000}      # BASELINE.json batch sizes
DEFAULT_TILE = {"C4": 1_000_000, "C5": 262144}      # syndromes per launch where the batch is tiled / streamed


def workload_spec(args, pkg):
    H, per, mi = pkg.codes.config_matrix(args.workload)
    per = args.per if args.per is not None else DEFAULT_PER[args.workload]
    B = args.batch if args.batch is not None else DEFAULT_B[args.workload]
    if args.max_iters is not None:
        mi = args.max_iters
    return H, float(per), int(mi), int(B)


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.power = []
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # NVML missing: report it instead of inventing numbers
            self.err = repr(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(0.05)

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "NVML unavailable"}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": float(self.max_mhz),
                "reasons": sorted(self.reasons), "power_w_max": max(self.power) if self.power else None,
                "samples": len(self.samples)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


def ncu_record(workload, variant, kernel_rev):
    """The tracked ncu summary (profiles/*.json, written by tools/ncu_summary.py --json) of this workload's dominant
    kernel, newest round first.  None if no capture is committed -- never a literal.  Records name it by its "file"."""
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_*.json")), reverse=True):
        try:
            d = json.load(open(path))
        except Exception:
            continue
        if d.get("workload") == workload and d.get("variant", "exact") == variant and str(d.get("kernel_rev", "")) == str(kernel_rev):
            d["file"] = os.path.relpath(path, ROOT)
            return d
    return None


def cpu_baseline_leg(oracle, H, per, mi, seed, budget_s, nthreads, dense=False):
    """Time the CPU restatement on a bounded sample of the same workload."""
    probe = 2000 if H.shape[1] < 20000 else 64
    _, syn = oracle.sample(H, per, seed, 0, probe)
    t0 = time.perf_counter()
    oracle.batch_decode(H, per, mi, syn, nthreads=nthreads, dense=dense)
    dt = max(time.perf_counter() - t0, 1e-4)
    n = int(min(max(probe, probe * budget_s / dt), 4_000_000))
    n = max(32, n // 32 * 32)
    _, syn = oracle.sample(H, per, seed, 0, n)
    t0 = time.perf_counter()
    r = oracle.batch_decode(H, per, mi, syn, nthreads=nthreads, dense=dense)
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": UNIT, "cores": int(nthreads), "kind": "port",
            "sample": "first %d syndromes of the same Philox stream, %s storage, %.2f s, mean iters %.3f" % (
                n, "dense s*n (faithful cost)" if dense else "edge-indexed", dt, float(r["iters"].mean()))}


def config_dict(args, H, per, mi, B, extra=None):
    s, n = H.shape
    d = {"workload": "%s: %s, s=%d n=%d E=%d, per=%g, max_iters=%d, batch=%d syndromes%s, early stop as reference" % (
        args.workload, WORKLOAD_NAMES[args.workload], s, n, H.nnz, per, mi, B, "" if getattr(args, "single_process", False) else "/GPU"),
        "per": per, "max_iters": mi, "batch_per_gpu": B, "variant": getattr(args, "variant", "exact"),
        "l2": "inputs+outputs of one step exceed the 126 MB L2" if B * ((s + 31) // 32 + (n + 31) // 32) * 4 > 130e6
        else "L2 flushed between steps (256 MB write)"}
    if extra:
        d.update(extra)
    return d


def run_reference(args):
    """--impl reference: the restated reference on the host cores (Julia is not installed on
    the box, so oracle/ is the reference arm; PARITY UNPINNED, see oracle/bp_oracle.c)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    pkg = entry.load_package()
    oracle = entry.load_oracle()
    oracle.build()
    H, per, mi, B = workload_spec(args, pkg)
    nthreads = oracle.num_threads()
    # size one step to ~2 s of wall time
    probe = 4096 if H.shape[1] < 20000 else 64
    _, syn = oracle.sample(H, per, SEED_E, 0, probe)
    oracle.batch_decode(H, per, mi, syn, nthreads=nthreads)          # spins the thread pool up
    t0 = time.perf_counter()
    oracle.batch_decode(H, per, mi, syn, nthreads=nthreads)
    dt = max(time.perf_counter() - t0, 1e-4)
    n = int(min(B, max(probe, probe * 2.0 / dt))) // 32 * 32
    n = max(n, 32)
    _, syn = oracle.sample(H, per, SEED_E, 0, n)
    for _ in range(args.warmup):
        oracle.batch_decode(H, per, mi, syn, nthreads=nthreads)
    t0 = time.perf_counter()
    iters_mean = 0.0
    for _ in range(args.steps):
        r = oracle.batch_decode(H, per, mi, syn, nthreads=nthreads)
        iters_mean = float(r["iters"].mean())
    dt = time.perf_counter() - t0
    value = n * args.steps / dt
    sample = "each step = first %d syndromes of the workload's Philox stream, edge-indexed restatement, %d threads, mean iters %.3f" % (
        n, nthreads, iters_mean)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "strong" if args.single_process else "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": config_dict(args, H, per, mi, B),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": nthreads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


_REAL_STDOUT = None


def protect_stdout():
    """Everything libraries print (NCCL banners, warnings) goes to stderr; stdout carries exactly
    the one JSON line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


# Extra operating points and the other configs' sub-records: a second JSON line on stderr, so that the result line keeps
# to the headline and stays a few KB (tools that read a command's output tail cannot parse a line of tens of KB).
DETAIL_KEYS = ("e2e_by_format", "sweep", "minsum", "fast32", "bposd_osd0", "config_C2_surface_d15_1M", "config_C4_hgp1600_10M",
               "config_C5_gallager100k_1M")


def emit(line):
    detail = {k: line.pop(k) for k in DETAIL_KEYS if k in line}
    if detail:
        sys.stderr.write(json.dumps({"detail": detail}) + "\n")
        sys.stderr.flush()
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


class DeviceRun:
    """HBM-resident decode loop of one decoder: synthetic syndromes of the whole batch generated on the device
    (Philox stream keyed by the global syndrome index), decoded in launches of `tile` syndromes."""

    def __init__(self, torch, dev, stream, dec, B, tile=None, first=0, seed=SEED_E):
        self.torch, self.dev, self.stream, self.dec = torch, dev, stream, dec
        self.B = int(B)
        self.tile = int(min(tile or B, B))
        self.first, self.seed = int(first), seed
        info = dec.info()
        self.info = info
        self.SW, self.NW = info["syn_words"], info["err_words"]
        self.st = stream.cuda_stream
        i32 = torch.int32
        self.synw = torch.empty((self.B, self.SW), dtype=i32, device=dev)
        # true errors / decoded errors / flags of ONE tile are kept (the batch streams through them)
        self.truth = torch.empty((self.tile, self.NW), dtype=i32, device=dev)
        self.errw = torch.empty((self.tile, self.NW), dtype=i32, device=dev)
        self.conv = torch.empty(self.tile, dtype=torch.uint8, device=dev)
        self.iters = torch.empty(self.tile, dtype=i32, device=dev)
        self.ctr = torch.zeros(4, dtype=torch.int64, device=dev)
        # the decoding kernel's own time: CUDA events recorded by the library on the launching stream around each launch
        dec.set_option("time_kernels", 1)
        self.kernel_s, self.kernel_launches = None, 0

    def sample(self, per):
        for t0 in range(0, self.B, self.tile):
            bt = min(self.tile, self.B - t0)
            self.dec.sample_device(bt, self.first + t0, self.seed, per, self.truth.data_ptr(), self.synw[t0:].data_ptr(), stream=self.st)

    def decode_once(self, ctr=None, B=None):
        B = self.B if B is None else B
        for t0 in range(0, B, self.tile):
            bt = min(self.tile, B - t0)
            self.dec.decode_device(bt, self.synw[t0:].data_ptr(), self.errw.data_ptr(), self.conv.data_ptr(), self.iters.data_ptr(),
                                   None, (ctr if ctr is not None else self.ctr).data_ptr(), stream=self.st)

    def timed(self, steps, warmup, flush=None, allreduce=None, barrier=None, warm_one_tile=False):
        """W warm-ups then `steps` timed decodes of the whole batch; CUDA events on the launching stream.
        Returns (seconds, summed counters, launches).  warm_one_tile: a warm-up step decodes one launch's worth
        (long streamed batches: the kernel, clocks and caches are warm after that)."""
        torch = self.torch
        for _ in range(warmup):
            self.ctr.zero_()
            self.decode_once(B=self.tile if warm_one_tile else None)
            if allreduce:
                allreduce(self.ctr)
        (barrier or torch.cuda.synchronize)()
        self.dec.kernel_time(reset=True)
        l0 = self.dec.launch_count()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        total = torch.zeros(4, dtype=torch.int64, device=self.dev)
        for a, b in evs:
            if flush is not None:
                flush.fill_(1)
            self.ctr.zero_()
            a.record(self.stream)
            self.decode_once()
            if allreduce:
                allreduce(self.ctr)            # the path's only collective: 4 int64 counters
            b.record(self.stream)
            total += self.ctr
        (barrier or torch.cuda.synchronize)()
        secs = sum(a.elapsed_time(b) for a, b in evs) / 1e3
        kms, kl = self.dec.kernel_time(reset=True)
        self.kernel_s, self.kernel_launches = kms / 1e3, kl       # summed over the timed steps
        return secs, total.cpu().numpy(), self.dec.launch_count() - l0

    def dump_last_step(self, out_dir, n, max_bytes=56 << 20):
        """What the last timed step returned to its caller, as .npy files in out_dir: for a fixed, seeded sample of the
        syndromes of the last tile decoded, their global indices, decoded errors (one row per syndrome), converged flags
        and iteration counts, plus the whole step's counters (decoded, converged, iterations).  The sample keeps the
        files under max_bytes."""
        torch = self.torch
        t0 = (self.B - 1) // self.tile * self.tile
        bt = self.B - t0
        k = int(min(bt, 65536, max(1, max_bytes // (4 * (n + 2) + 8))))
        local = np.sort(np.random.default_rng(SEED_E).choice(bt, size=k, replace=False))
        idx = torch.from_numpy(local).to(self.dev)
        torch.cuda.synchronize()
        words = self.errw[idx].cpu().numpy().view(np.uint8)            # bit r % 32 of little-endian word r / 32
        errors = np.unpackbits(words, axis=1, bitorder="little")[:, :n]
        os.makedirs(out_dir, exist_ok=True)
        out = {"syndrome_index": (self.first + t0 + local).astype(np.float64),
               "errors": errors.astype(np.float32),
               "converged": self.conv[idx].cpu().numpy().astype(np.float32),
               "iterations": self.iters[idx].cpu().numpy().astype(np.float32),
               "counters": self.ctr[:3].cpu().numpy().astype(np.float64)}
        for name, a in out.items():
            np.save(os.path.join(out_dir, name + ".npy"), a)

    def exact_match_frac_last_tile(self, per):
        """Exact-match fraction of the LAST tile decoded (its true errors are regenerated from the same stream)."""
        torch = self.torch
        score = torch.zeros(2, dtype=torch.int64, device=self.dev)
        t0 = (self.B - 1) // self.tile * self.tile
        bt = self.B - t0
        self.dec.sample_device(bt, self.first + t0, self.seed, per, self.truth.data_ptr(), self.synw[t0:].data_ptr(), stream=self.st)
        self.dec.score_device(bt, self.truth.data_ptr(), self.errw.data_ptr(), self.synw[t0:].data_ptr(), score.data_ptr(), stream=self.st)
        torch.cuda.synchronize()
        return float(score[0].item()) / bt


def roofline_of(info, variant, E, SW, NW, B_per_step_gpu, units_per_step_gpu, step_s, clk_mhz, peaks, peaks_src, ncu,
                kernel_s=None, kernel_launches=0, filtered_per_step=0.0):
    """Roofline object of the dominant kernel (this rank's share, this rank's time).
    kernel_s: that kernel's own time per step (CUDA events on the launching stream around each of its launches, recorded by
    the library: option time_kernels); filtered_per_step: syndromes the first-iteration filter finished (their single
    iteration never reaches the decoding kernel).  achieved = algorithmic work of the kernel's launches / the kernel's time;
    the whole-step figure (all kernels of the step, the filter's savings counted as work done) is reported next to it."""
    io_bytes = B_per_step_gpu * (SW * 4 + NW * 4 + 1 + 4)
    alg_bytes = units_per_step_gpu * 4.0 * E * 8.0 + io_bytes
    k_s = kernel_s if kernel_s and kernel_s > 0 else step_s
    k_units = max(units_per_step_gpu - filtered_per_step, 0.0)
    timing = {"kernel_ms_per_step": 1e3 * k_s, "kernel_launches_per_step": kernel_launches, "step_ms": 1e3 * step_s,
              "kernel_share_of_step": k_s / step_s, "kernel_units_per_step": k_units, "step_units_per_step": units_per_step_gpu,
              "how": "CUDA events on the launching stream around every launch of the decoding kernel" if kernel_s else "step time (kernel not timed separately)"}
    traffic = None
    if ncu and ncu.get("dram_bytes_read") is not None and ncu.get("syndromes"):
        # DRAM bytes of the profiled launch, per launch of this run (both are linear in the launch's batch)
        per_syn = (ncu["dram_bytes_read"] + ncu["dram_bytes_write"]) / float(ncu["syndromes"])
        traffic = per_syn * B_per_step_gpu / max(kernel_launches, 1)
    if info["family"] == 1:
        slots = FP64_SLOTS[variant]
        peak = info["sm_count"] * FP64_LANES_PER_SM_CLK * clk_mhz * 1e6 / 1e12
        ach = k_units * E * slots["model"] / k_s / 1e12
        roof = {"bound": "fp64", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                "frac_model_%d" % slots["model"]: ach / peak,
                "frac_executed_%d" % slots["executed"]: k_units * E * slots["executed"] / k_s / 1e12 / peak,
                "whole_step_frac_model_%d" % slots["model"]: units_per_step_gpu * E * slots["model"] / step_s / 1e12 / peak,
                "traffic": traffic, "timing": timing,
                "note": "shared-memory-resident kernel: bounded by the FP64 pipe, not HBM or tensor cores. achieved = (syndrome, iteration) pairs the "
                        "decoding kernel executed (the step's minus the single iterations the first-iteration filter finished with integer "
                        "instructions) x E x %d FP64-pipe issue slots per edge-iteration of the %s arithmetic / the kernel's own CUDA-event time; "
                        "frac_executed counts the %d the kernel issues (comparable with ncu's sm__pipe_fp64_cycles_active); whole_step_frac counts "
                        "every iteration of the step against the step time (the filter's iterations cost no FP64 work, so it is a speed-up "
                        "figure, not a pipe utilisation); peak = %d SMs x 64 FP64 lanes/clk x median SM clock under load (%.0f MHz); one FLOP = "
                        "one FP64 lane-instruction" % (
                            slots["model"], "reference" if variant == "exact" else variant, slots["executed"], info["sm_count"], clk_mhz),
                "ncu": ncu and ncu["file"],
                "hbm_model": {"achieved_GBps": alg_bytes / step_s / 1e9, "peak_GBps": peaks["hbm_gbs"], "peak_source": peaks_src,
                              "frac": alg_bytes / step_s / 1e9 / peaks["hbm_gbs"],
                              "note": "4*E*8 B per syndrome-iteration if messages lived in HBM (they live in shared memory) + packed I/O"}}
    else:
        ach = alg_bytes / k_s / 1e9
        roof = {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": ach / peaks["hbm_gbs"], "whole_step_frac": alg_bytes / step_s / 1e9 / peaks["hbm_gbs"],
                "traffic": traffic, "timing": timing,
                "algorithmic_bytes_per_step": alg_bytes,
                "algorithmic_bytes_per_launch": alg_bytes / max(kernel_launches, 1),
                "note": "algorithmic bytes = 4*E*8 per syndrome-iteration + packed I/O of the kernel's launches / the kernel's own CUDA-event time; "
                        "peak = %s copy bandwidth; message store %d MB per GPU; traffic = ncu dram bytes of one profiled launch scaled to this "
                        "run's launch size" % (peaks_src, info["message_bytes"] >> 20),
                "ncu": ncu and ncu["file"]}
    return roof


def sub_record(pkg, torch, dev, stream, name, per, B, tile, steps, warmup, peaks, peaks_src, clk_mhz, oracle=None, cpu_budget=3.0,
               variant="exact", **opts):
    """One BASELINE config next to the headline: HBM-resident throughput at its full batch size, roofline, CPU baseline."""
    H, _, mi = pkg.codes.config_matrix(name)
    dec = pkg.BeliefPropagationDecoder(H, per, mi, devices=[dev.index], variant=variant, **opts)
    run = DeviceRun(torch, dev, stream, dec, B, tile)
    run.sample(per)
    secs, c, launches = run.timed(steps, warmup, warm_one_tile=run.tile < B)
    info = run.info
    rec = {"workload": "%s: %s, s=%d n=%d E=%d, per=%g, max_iters=%d, batch=%d%s" % (
        name, WORKLOAD_NAMES[name], H.shape[0], H.shape[1], H.nnz, per, mi, B,
        "" if run.tile >= B else " streamed from HBM in launches of %d" % run.tile),
        "per": per, "value": float(c[0]) / secs, "unit": UNIT, "steps": steps, "warmup": warmup, "ms_per_step": 1e3 * secs / steps,
        "mean_iters": float(c[2]) / max(float(c[0]), 1.0), "converged_frac": float(c[1]) / max(float(c[0]), 1.0),
        "syndrome_iterations_per_s": float(c[2]) / secs, "gpu_launches": int(launches),
        "kernel": {k: info[k] for k in ("family", "kernel_mode", "ctas_per_sm", "threads_per_cta", "message_bytes", "prefetch_distance", "kernel_rev")}}
    rec["roofline"] = roofline_of(info, variant, H.nnz, run.SW, run.NW, B, float(c[2]) / steps, secs / steps, clk_mhz, peaks, peaks_src,
                                  ncu_record(name, variant, info["kernel_rev"]),
                                  kernel_s=run.kernel_s / steps, kernel_launches=run.kernel_launches / steps, filtered_per_step=float(c[3]) / steps)
    if oracle is not None:
        rec["cpu_baseline"] = cpu_baseline_leg(oracle, H, per, mi, SEED_E, cpu_budget, oracle.num_threads())
    dec.close()
    del run
    torch.cuda.empty_cache()
    return rec


def host_bitmatrix(torch, dev, synw, s, B, pinned):
    """Host BitMatrix (bit c*s + r of a little-endian stream) of the packed device rows synw[:B]."""
    nb = (B * s + 63) // 64 * 8
    bit_ar = torch.arange(s, device=dev, dtype=torch.int64)
    weights = (2 ** torch.arange(8, device=dev, dtype=torch.int32)).to(torch.uint8)
    acc = torch.zeros(nb * 8, dtype=torch.uint8, device=dev)
    sl = 1 << 19
    for b0 in range(0, B, sl):
        w = synw[b0:min(b0 + sl, B)].to(torch.int64) & 0xFFFFFFFF
        bits = ((w[:, bit_ar // 32] >> (bit_ar % 32)) & 1).to(torch.uint8)       # [rows, s]
        acc[b0 * s:(b0 + bits.shape[0]) * s] = bits.reshape(-1)
        del w, bits
    d_bits = (acc.view(-1, 8) * weights).sum(dim=1, dtype=torch.int32).to(torch.uint8)
    del acc
    h = torch.empty(nb, dtype=torch.uint8, pin_memory=pinned)
    h.copy_(d_bits)
    torch.cuda.synchronize()
    return h


def e2e_leg(dec, B, np_in, fmt_in, ld_in, np_out, fmt_out, ld_out, np_conv, steps, barrier, warm=2):
    for _ in range(warm):
        dec.decode_raw(B, np_in, fmt_in, ld_in, np_out, fmt_out, ld_out, np_conv)
    barrier()
    l0 = dec.launch_count()
    t0 = time.perf_counter()
    for _ in range(steps):
        dec.decode_raw(B, np_in, fmt_in, ld_in, np_out, fmt_out, ld_out, np_conv)
    barrier()
    return time.perf_counter() - t0, dec.launch_count() - l0


def main():
    protect_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C3", choices=["C1", "C2", "C3", "C4", "C5"])
    ap.add_argument("--per", type=float, default=None)
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--tile", type=int, default=None, help="syndromes per launch (C4 / C5 stream their batch through HBM in tiles)")
    ap.add_argument("--max-iters", type=int, default=None, dest="max_iters")
    ap.add_argument("--no-sweep", action="store_true", help="skip the extra operating points and the C2/C4/C5 sub-records")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--single-process", action="store_true", dest="single_process",
                    help="ONE decoder on devices 0..N-1 (in-library sharding, std::thread per device), one host batch: strong scaling")
    ap.add_argument("--family", type=int, default=0)
    ap.add_argument("--warps", type=int, default=0)
    ap.add_argument("--prefetch", type=int, default=-1)
    ap.add_argument("--kernel-profile", action="store_true", dest="kernel_profile",
                    help="phase timing of the shared-memory kernel (adds clock reads; not a bench value)")
    ap.add_argument("--max-ctas", type=int, default=0, dest="max_ctas", help="cap on resident CTAs per SM (experiments)")
    ap.add_argument("--lean", type=int, default=-1, help="family SMEM: 1 = round-2 kernel (default), 0 = general persistent kernel")
    ap.add_argument("--strong", action="store_true",
                    help="under torchrun: ONE batch of the workload's size split over the ranks (sharding.shard_range) instead of "
                         "one batch per rank: strong scaling of the one-process-per-GPU form")
    ap.add_argument("--opt", action="append", default=[], metavar="KEY=VALUE",
                    help="extra ldpcb200_set_option pairs (experiments), e.g. --opt dual=1")
    ap.add_argument("--variant", default="exact", choices=["exact", "minsum", "fast"],
                    help="exact = reference-parity sum-product (headline); minsum = normalised min-sum (no reference equivalent)")
    ap.add_argument("--dump-outputs", default=None, dest="dump_outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (a seeded sample of "
                         "the decoded syndromes, at most 64 MB), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.single_process):
        ap.error("--dump-outputs applies to the device-resident run (--impl ours without --single-process)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback (use --impl reference for the CPU arm)")
    if args.single_process:
        if world > 1 and rank != 0:          # launched under torchrun: rank 0 alone owns all devices
            return
        return run_single_process(args, torch)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    entry.build()
    pkg = entry.load_package()
    lib = pkg._lib
    H, per, mi, B = workload_spec(args, pkg)
    s, n = H.shape
    E = H.nnz
    opts = {}
    if args.family:
        opts["family"] = args.family
    if args.warps:
        opts["warps"] = args.warps
    if args.prefetch >= 0:
        opts["prefetch"] = args.prefetch
    if args.lean >= 0:
        opts["lean"] = args.lean
    if args.max_ctas > 0:
        opts["max_ctas_per_sm"] = args.max_ctas
    if args.kernel_profile:
        opts["kernel_profile"] = 1
    for kv in args.opt:
        k, v = kv.split("=", 1)
        opts[k] = int(v)
    dec = pkg.BeliefPropagationDecoder(H, per, mi, devices=[local], variant=args.variant, **opts)
    # a non-default torch stream: its handle is non-NULL, so the library launches on exactly the
    # stream the torch CUDA events are recorded on (NULL would mean "the handle's own stream")
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    tile = args.tile if args.tile is not None else DEFAULT_TILE.get(args.workload)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    allreduce = pkg.sharding.allreduce_counters if world > 1 else None     # the path's only collective
    B_total, first = B * world, rank * B                   # weak scaling: every rank owns global syndromes [r*B, (r+1)*B)
    if args.strong and world > 1:                          # strong scaling: one batch, contiguous 32-aligned column ranges
        B_total = B
        first, hi = pkg.sharding.shard_range(B_total, rank, world)
        B = hi - first
    # ---- synthetic inputs, resident in HBM; shard r owns global syndromes [r*B, (r+1)*B)
    run = DeviceRun(torch, dev, stream, dec, B, tile, first=first)
    info = run.info
    SW, NW = run.SW, run.NW
    flush = None
    if B * (SW + NW) * 4 <= 130e6:
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    run.sample(per)
    run.timed(0, args.warmup, flush, allreduce, barrier)
    sampler = ClockSampler(local)
    sampler.start()                               # clocks are sampled during the timed region only
    secs, c, launches = run.timed(args.steps, 0, flush, allreduce, barrier)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        run.dump_last_step(args.dump_outputs, n)
    t = torch.tensor([secs], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    secs = float(t.item())
    n_dec_all = float(c[0])                       # all ranks (counters were all-reduced), all steps
    value = n_dec_all / secs
    mean_iters = float(c[2]) / max(float(c[0]), 1.0)
    conv_frac = float(c[1]) / max(float(c[0]), 1.0)
    exact_frac = run.exact_match_frac_last_tile(per)

    # ---- roofline of the dominant kernel (this rank's share, this rank's time)
    peaks, peaks_src = measured_peaks()
    units_per_step_gpu = float(c[2]) / args.steps / world           # (syndrome, iteration) pairs per step per GPU
    step_s = secs / args.steps
    clk_mhz = clocks.get("sm_mhz") or peaks.get("sm_max_mhz", 1965.0)
    roof = roofline_of(info, args.variant, E, SW, NW, B, units_per_step_gpu, step_s, clk_mhz, peaks, peaks_src,
                       ncu_record(args.workload, args.variant, info["kernel_rev"]),
                       kernel_s=run.kernel_s / args.steps, kernel_launches=run.kernel_launches / args.steps,
                       filtered_per_step=float(c[3]) / args.steps / world)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * step_s, "higher_is_better": True, "scaling": "strong" if (args.strong and world > 1) else "weak",
            "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": config_dict(args, H, per, mi, B, dict({"tile": run.tile} if run.tile < B else {}, batch_total=B_total,
                                                             split="one batch split over the ranks (strong)" if (args.strong and world > 1)
                                                             else "one batch per rank (weak)")),
            "mean_iters": mean_iters, "converged_frac": conv_frac, "exact_match_frac": exact_frac,
            "syndrome_iterations_per_s": float(c[2]) / secs,
            "roofline": roof, "gpu_launches": int(launches), "clocks": clocks,
            "kernel": {k: info[k] for k in ("family", "kernel_mode", "ctas_per_sm", "threads_per_cta", "smem_bytes", "slots",
                                            "message_bytes", "prefetch_distance", "kernel_rev")}}
    if args.kernel_profile:
        kp = dec.kernel_profile()
        wi = max(kp["warp_iterations"], 1)
        line["kernel_profile_cycles_per_warp_iteration"] = {k: round(v / wi, 1) for k, v in kp.items() if k != "warp_iterations"}

    # ---- end to end through the host-buffer C-ABI call
    if not args.no_e2e:
        Be = int(min(B, 10_000_000))
        e2e_steps = max(2, min(args.steps, 5))
        conv_dev_count = None
        if world == 1:          # converged count of the same syndromes from the device-resident path
            cchk = torch.zeros(4, dtype=torch.int64, device=dev)
            run.decode_once(cchk, Be)
            torch.cuda.synchronize()
            conv_dev_count = int(cchk[1].item())
        h_in = host_bitmatrix(torch, dev, run.synw, s, Be, pinned=True)
        nb_out = (Be * n + 63) // 64 * 8
        h_out = torch.empty(nb_out, dtype=torch.uint8, pin_memory=True)
        h_conv = torch.empty(Be, dtype=torch.uint8, pin_memory=True)
        np_in, np_out, np_conv = h_in.numpy(), h_out.numpy(), h_conv.numpy()
        dt, nl = e2e_leg(dec, Be, np_in, lib.FMT_BITS, 0, np_out, lib.FMT_BITS, 0, np_conv, e2e_steps, barrier)
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
        line["e2e"] = {"value": world * Be * e2e_steps / dt, "unit": UNIT, "h2d_bytes_per_step": int(h_in.numel()),
                       "d2h_bytes_per_step": int(nb_out + Be), "steps": e2e_steps, "batch_per_gpu": Be,
                       "api": "ldpcb200_decode_batch(FMT_BITS in/out = Julia BitMatrix, pinned host buffers), wall clock around the blocking call",
                       "converged_check": (int(np_conv.sum()) == conv_dev_count) if conv_dev_count is not None else None,
                       "gpu_launches": int(nl)}
        if world == 1 and not args.no_sweep and args.workload in ("C2", "C3"):
            # the same call with the buffers a Julia caller really has: pageable arrays, and the Matrix{Int} syndromes of
            # the reference's own test (test/test_bp_decoder.jl:24-26: batchdecode!(bpd, syndromes::Matrix{Int}, zero(errors)::BitMatrix))
            table = [{"in": "BitMatrix", "out": "BitMatrix", "host_memory": "pinned", "batch": Be, "value": line["e2e"]["value"],
                      "h2d_bytes": int(h_in.numel()), "d2h_bytes": int(nb_out + Be)}]
            pg_in = np.array(np_in, copy=True)            # ordinary (pageable) numpy memory
            pg_out = np.zeros(nb_out, dtype=np.uint8)
            pg_conv = np.zeros(Be, dtype=np.uint8)
            dt, _ = e2e_leg(dec, Be, pg_in, lib.FMT_BITS, 0, pg_out, lib.FMT_BITS, 0, pg_conv, e2e_steps, barrier)
            ok = bool(np.array_equal(pg_out, np_out) and np.array_equal(pg_conv, np_conv))
            table.append({"in": "BitMatrix", "out": "BitMatrix", "host_memory": "pageable", "batch": Be, "value": Be * e2e_steps / dt,
                          "h2d_bytes": int(pg_in.size), "d2h_bytes": int(nb_out + Be), "same_outputs_as_pinned": ok})
            Bi = int(min(Be, 2_000_000))                  # Matrix{Int}: 8 bytes per syndrome bit -> a 2M-column sample (1.2 GB)
            st2 = max(2, e2e_steps // 2)
            bits = np.unpackbits(np_in[: (Bi * s + 7) // 8], bitorder="little")[: Bi * s]
            syn_i64 = np.asfortranarray(bits.reshape(Bi, s).T.astype(np.int64))
            out_b = np.zeros((Bi * n + 63) // 64 * 8, dtype=np.uint8)
            cv_b = np.zeros(Bi, dtype=np.uint8)
            dt, _ = e2e_leg(dec, Bi, syn_i64, lib.FMT_I64, s, out_b, lib.FMT_BITS, 0, cv_b, st2, barrier, warm=1)
            nb = Bi * n // 8
            table.append({"in": "Matrix{Int}", "out": "BitMatrix", "host_memory": "pageable", "batch": Bi,
                          "value": Bi * st2 / dt, "h2d_bytes": int(syn_i64.nbytes), "d2h_bytes": int(out_b.size + Bi),
                          "same_outputs_as_pinned": bool(np.array_equal(out_b[:nb], np_out[:nb]) and np.array_equal(cv_b, np_conv[:Bi])),
                          "note": "the call of test/test_bp_decoder.jl:24-26; 8 bytes of PCIe traffic per syndrome bit"})
            syn_u8 = np.asfortranarray(bits.reshape(Bi, s).T.astype(np.uint8))
            out_u8 = np.zeros((n, Bi), dtype=np.uint8, order="F")
            dt, _ = e2e_leg(dec, Bi, syn_u8, lib.FMT_U8, s, out_u8, lib.FMT_U8, n, cv_b, st2, barrier, warm=1)
            table.append({"in": "Matrix{Bool}", "out": "Matrix{Bool}", "host_memory": "pageable", "batch": Bi,
                          "value": Bi * st2 / dt, "h2d_bytes": int(syn_u8.nbytes), "d2h_bytes": int(out_u8.nbytes + Bi)})
            line["e2e_by_format"] = table
            del pg_in, pg_out, syn_i64, syn_u8, out_u8, out_b, bits
        del h_in, h_out, h_conv

    # ---- extra operating points of the headline code (not the headline): per sweep, forced max_iters, min-sum
    if world == 1 and not args.no_sweep and args.workload in ("C2", "C3") and args.variant == "exact":
        sweep = []
        for p_ in ([0.001, 0.01, 0.03, 0.1] if args.workload == "C3" else [0.001, 0.003, 0.01, 0.03, 0.1]):
            d2 = pkg.BeliefPropagationDecoder(H, p_, mi, devices=[local], **opts)
            r2 = DeviceRun(torch, dev, stream, d2, B)
            r2.sample(p_)
            secs2, c2, _ = r2.timed(3, 1, flush)
            sweep.append({"per": p_, "value": float(c2[0]) / secs2, "mean_iters": float(c2[2]) / float(c2[0]),
                          "converged_frac": float(c2[1]) / float(c2[0]), "syndrome_iterations_per_s": float(c2[2]) / secs2})
            d2.close()
            del r2
        # forced iterations: its own decoder, so that the library configures for that mode (early_stop = 0 before the
        # first decode)
        d2 = pkg.BeliefPropagationDecoder(H, per, mi, devices=[local], early_stop=0, **opts)
        r2 = DeviceRun(torch, dev, stream, d2, B)
        r2.sample(per)
        secs2, c2, _ = r2.timed(2, 1, flush)
        d2.close()
        del r2
        peak = info["sm_count"] * FP64_LANES_PER_SM_CLK * clk_mhz * 1e6 / 1e12
        sweep.append({"per": per, "forced_iters": mi, "value": float(c2[0]) / secs2, "mean_iters": float(c2[2]) / float(c2[0]),
                      "syndrome_iterations_per_s": float(c2[2]) / secs2,
                      "fp64_frac_model_26": float(c2[2]) * E * 26 / secs2 / 1e12 / peak,
                      "fp64_frac_executed_21": float(c2[2]) * E * 21 / secs2 / 1e12 / peak})
        line["sweep"] = sweep
        # sum-product vs min-sum (BASELINE.json config 3): the normalised min-sum kernels on the same syndromes; no
        # reference equivalent, so it is reported by quality, not parity
        errw_sp = run.errw.clone()
        dms = pkg.BeliefPropagationDecoder(H, per, mi, devices=[local], variant="minsum")
        rms = DeviceRun(torch, dev, stream, dms, B)
        rms.sample(per)
        secs2, c2_, _ = rms.timed(3, 2, flush)
        ms_info = rms.info
        differ = int((rms.errw != errw_sp).any(dim=1).sum().item()) if run.tile >= B else None
        ms_roof = roofline_of(ms_info, "minsum", E, SW, NW, B, float(c2_[2]) / 3, secs2 / 3, clk_mhz, peaks, peaks_src,
                              ncu_record(args.workload, "minsum", ms_info["kernel_rev"]),
                              kernel_s=rms.kernel_s / 3, kernel_launches=rms.kernel_launches / 3, filtered_per_step=float(c2_[3]) / 3)
        line["minsum"] = {"value": float(c2_[0]) / secs2, "unit": UNIT, "per": per, "scale": 0.875,
                          "mean_iters": float(c2_[2]) / float(c2_[0]), "converged_frac": float(c2_[1]) / float(c2_[0]),
                          "exact_match_frac": rms.exact_match_frac_last_tile(per),
                          "decisions_differ_from_sum_product_frac": differ / B if differ is not None else None,
                          "roofline": {k: ms_roof[k] for k in ms_roof if k not in ("note", "hbm_model")},
                          "note": "FP64 log-likelihood-ratio min-sum, same schedule/early stop; sum-product exact_match_frac is the line's own; "
                                  "5 FP64-pipe slots per edge-iteration (no divisions): the kernel is issue/shared-memory bound, not FP64 bound"}
        dms.close()
        del rms
        # the fast FP32 tanh/atanh variant (north star; SURVEY K6): quality against the exact kernels on the same syndromes
        dfa = pkg.BeliefPropagationDecoder(H, per, mi, devices=[local], variant="fast")
        rfa = DeviceRun(torch, dev, stream, dfa, B)
        rfa.sample(per)
        secs3, c3_, _ = rfa.timed(3, 2, flush)
        differ = int((rfa.errw != errw_sp).any(dim=1).sum().item()) if run.tile >= B else None
        line["fast32"] = {"value": float(c3_[0]) / secs3, "unit": UNIT, "per": per,
                          "mean_iters": float(c3_[2]) / float(c3_[0]), "converged_frac": float(c3_[1]) / float(c3_[0]),
                          "exact_match_frac": rfa.exact_match_frac_last_tile(per),
                          "decisions_differ_from_exact_frac": differ / B if differ is not None else None,
                          "kernel": {k: rfa.info[k] for k in ("family", "kernel_mode", "ctas_per_sm", "threads_per_cta", "kernel_rev")},
                          "note": "FP32 log-likelihood-ratio tanh/atanh sum-product with MUFU EX2/RCP/LG2, same schedule/early stop; messages "
                                  "travel through the same 8-byte shared-memory slots (kernel structure shared with the exact variant); "
                                  "not bit-compatible with the reference: compare exact_match_frac / converged_frac with the line's own"}
        dfa.close()
        del errw_sp, rfa

    # ---- BASELINE.json config 4 is "the BP stage of BP+OSD": the whole BP -> OSD-0 pipeline on the same syndromes
    # (ldpcb200_decode_device with posterior ratios, then ldpcb200_osd0_device on the unconverged ones)
    if world == 1 and not args.no_sweep and args.workload == "C4" and args.variant == "exact":
        line["bposd_osd0"] = bposd_record(args, pkg, torch, dev, stream, dec, run, H, per, mi, n, SW, NW)

    # ---- the other BASELINE configs next to the headline at their full batch sizes (N = 1, default workload only)
    if world == 1 and not args.no_sweep and args.workload == "C3" and args.variant == "exact":
        oracle = None if args.no_cpu else entry.load_oracle()
        del run
        run = None
        torch.cuda.empty_cache()
        c2rec = []
        for p_ in (0.001, 0.003, 0.01, 0.03, 0.1):
            c2rec.append(sub_record(pkg, torch, dev, stream, "C2", p_, DEFAULT_B["C2"], None, 5, 3, peaks, peaks_src, clk_mhz,
                                    oracle=oracle if p_ == 0.01 else None, cpu_budget=2.0))
        line["config_C2_surface_d15_1M"] = c2rec
        line["config_C4_hgp1600_10M"] = sub_record(pkg, torch, dev, stream, "C4", DEFAULT_PER["C4"], DEFAULT_B["C4"], DEFAULT_TILE["C4"], 2, 3,
                                                   peaks, peaks_src, clk_mhz, oracle=oracle, cpu_budget=3.0)
        line["config_C5_gallager100k_1M"] = sub_record(pkg, torch, dev, stream, "C5", DEFAULT_PER["C5"], DEFAULT_B["C5"], DEFAULT_TILE["C5"], 1, 3,
                                                       peaks, peaks_src, clk_mhz, oracle=oracle, cpu_budget=3.0)

    # ---- CPU baseline next to it (rank 0, N = 1 only)
    if rank == 0 and world == 1 and not args.no_cpu:
        oracle = entry.load_oracle()
        line["cpu_baseline"] = cpu_baseline_leg(oracle, H, per, mi, SEED_E, 10.0, 1)
        line["cpu_baseline_all_threads"] = cpu_baseline_leg(oracle, H, per, mi, SEED_E, 5.0, oracle.num_threads())
        if s * n * 16 < 2e9:
            line["cpu_baseline_dense_faithful"] = cpu_baseline_leg(oracle, H, per, mi, SEED_E, 5.0, 1, dense=True)
    dec.close()
    if rank == 0:
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def bposd_record(args, pkg, torch, dev, stream, dec, run, H, per, mi, n, SW, NW):
    st = stream.cuda_stream
    Bo = int(min(run.tile, 131072))
    synw, errw, conv, iters, ctr, truth = run.synw, run.errw, run.conv, run.iters, run.ctr, run.truth
    ratio = torch.empty((Bo, n), dtype=torch.float64, device=dev)
    stats = torch.zeros(8, dtype=torch.int64, device=dev)
    sc_bp = torch.zeros(2, dtype=torch.int64, device=dev)
    sc_osd = torch.zeros(2, dtype=torch.int64, device=dev)
    dec.sample_device(Bo, run.first, SEED_E, per, truth.data_ptr(), synw.data_ptr(), stream=st)

    def bp_stage():
        dec.decode_device(Bo, synw.data_ptr(), errw.data_ptr(), conv.data_ptr(), iters.data_ptr(), ratio.data_ptr(),
                          ctr.data_ptr(), stream=st)

    def osd_stage():
        dec.osd0_device(Bo, synw.data_ptr(), errw.data_ptr(), conv.data_ptr(), ratio.data_ptr(), stats.data_ptr(), stream=st)

    dec.set_option("ratio_last_only", 1)
    for _ in range(2):
        bp_stage()
        osd_stage()
    torch.cuda.synchronize()
    reps = 3
    t_bp = t_osd = 0.0
    stats.zero_()
    ctr.zero_()
    for rep in range(reps):
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record(stream)
        bp_stage()
        e1.record(stream)
        if rep == 0:
            dec.score_device(Bo, truth.data_ptr(), errw.data_ptr(), synw.data_ptr(), sc_bp.data_ptr(), stream=st)
            torch.cuda.synchronize()
        e1b = torch.cuda.Event(enable_timing=True)
        e1b.record(stream)
        osd_stage()
        e2.record(stream)
        torch.cuda.synchronize()
        t_bp += e0.elapsed_time(e1) / 1e3
        t_osd += e1b.elapsed_time(e2) / 1e3
    dec.score_device(Bo, truth.data_ptr(), errw.data_ptr(), synw.data_ptr(), sc_osd.data_ptr(), stream=st)
    torch.cuda.synchronize()
    so = stats.cpu().numpy()
    nproc = float(so[0]) / reps
    if os.environ.get("LDPCB200_OSD_PROFILE"):     # one extra pass with the kernel's per-phase cycle counters on
        dec.set_option("osd_profile", 1)
        stats.zero_()
        bp_stage()
        osd_stage()
        torch.cuda.synchronize()
        sp_ = stats.cpu().numpy()
        sys.stderr.write("osd phases (SM cycles per syndrome): sort %.0f build %.0f search %.0f update %.0f solve %.0f\n" %
                         tuple(float(sp_[k]) / max(float(sp_[0]), 1.0) for k in (3, 4, 5, 6, 7)))
        dec.set_option("osd_profile", 0)
    bposd = {"batch": Bo, "per": per, "value": Bo * reps / (t_bp + t_osd), "unit": UNIT,
             "bp_stage_syndromes_per_s": Bo * reps / t_bp,
             "osd_stage_syndromes_per_s": float(so[0]) / t_osd if t_osd > 0 else None,
             "osd_stage_ms": t_osd / reps * 1e3, "bp_stage_ms": t_bp / reps * 1e3,
             "unconverged_frac": nproc / Bo,
             "mean_pivots": float(so[1]) / max(float(so[0]), 1.0), "mean_columns_visited": float(so[2]) / max(float(so[0]), 1.0),
             "bp_exact_match_frac": float(sc_bp[0].item()) / Bo, "bp_syndrome_satisfied_frac": float(sc_bp[1].item()) / Bo,
             "bposd_exact_match_frac": float(sc_osd[0].item()) / Bo,
             "bposd_syndrome_satisfied_frac": float(sc_osd[1].item()) / Bo,
             "note": "device-resident; the BP stage writes posterior ratios only in iteration max_iters (ratio_last_only)"}
    if not args.no_e2e:
        # the reference-facing call: host arrays in, host arrays out (ldpcb200_bposd_decode_batch)
        syn_t = torch.empty((Bo, SW), dtype=torch.int32, pin_memory=True)
        syn_t.copy_(synw[:Bo])
        err_t = torch.zeros((Bo, NW), dtype=torch.int32, pin_memory=True)
        conv_t = torch.zeros(Bo, dtype=torch.uint8, pin_memory=True)
        torch.cuda.synchronize()
        syn_h, err_h, conv_h = syn_t.numpy().view(np.uint32), err_t.numpy().view(np.uint32), conv_t.numpy()
        dec.bposd_raw(Bo, syn_h, pkg._lib.FMT_PACKED32, SW, err_h, pkg._lib.FMT_PACKED32, NW, conv_h)
        t0 = time.perf_counter()
        for _ in range(reps):
            dec.bposd_raw(Bo, syn_h, pkg._lib.FMT_PACKED32, SW, err_h, pkg._lib.FMT_PACKED32, NW, conv_h)
        dt = time.perf_counter() - t0
        bposd["e2e"] = {"value": Bo * reps / dt, "unit": UNIT, "h2d_bytes_per_step": int(Bo * SW * 4),
                        "d2h_bytes_per_step": int(Bo * (NW * 4 + 1)),
                        "api": "ldpcb200_bposd_decode_batch(FMT_PACKED32 in/out, pinned host buffers), wall clock"}
    if not args.no_cpu:
        oracle = entry.load_oracle()
        nth = oracle.num_threads()
        Kc = 8 * nth
        _, syn_c = oracle.sample(H, per, SEED_E, 0, Kc)
        oracle.bposd_decode(H, per, mi, syn_c[:, :nth], nthreads=nth)
        t0 = time.perf_counter()
        oracle.bposd_decode(H, per, mi, syn_c, nthreads=nth)
        dt = time.perf_counter() - t0
        bposd["cpu_baseline"] = {"value": Kc / dt, "unit": UNIT, "cores": nth, "kind": "port",
                                 "sample": "first %d syndromes of the same stream, BP + restated OSD-0 (bit-packed rows)" % Kc}
    dec.set_option("ratio_last_only", 0)
    del ratio
    return bposd


def run_single_process(args, torch):
    """ONE decoder handle over devices 0..N-1: the call a Julia user makes with `devices = 0:N-1`.  The library splits
    the host batch into contiguous column ranges (std::thread per device, chunked double-buffered copies) and sums the
    counters (ncclAllReduce over its own communicators when NCCL is available).  The batch is FIXED (BASELINE config 3:
    one 10M-syndrome batch at 1/2/4/8 GPUs): strong scaling."""
    N = int(args.gpus)
    if torch.cuda.device_count() < N:
        raise SystemExit("--single-process --gpus %d needs %d visible devices (found %d)" % (N, N, torch.cuda.device_count()))
    entry.build()
    pkg = entry.load_package()
    lib = pkg._lib
    H, per, mi, B = workload_spec(args, pkg)
    s, n = H.shape
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    # reference run on device 0 alone, device-resident: converged count / iterations the sharded call must reproduce
    d0 = pkg.BeliefPropagationDecoder(H, per, mi, devices=[0], variant=args.variant)
    run = DeviceRun(torch, dev, stream, d0, B)
    run.sample(per)
    run.ctr.zero_()
    run.decode_once()
    torch.cuda.synchronize()
    want = run.ctr.cpu().numpy().copy()
    h_in = host_bitmatrix(torch, dev, run.synw, s, B, pinned=True)
    d0.close()
    del run
    torch.cuda.empty_cache()
    dec = pkg.BeliefPropagationDecoder(H, per, mi, devices=list(range(N)), variant=args.variant)
    info = dec.info()
    nb_out = (B * n + 63) // 64 * 8
    h_out = torch.empty(nb_out, dtype=torch.uint8, pin_memory=True)
    h_conv = torch.empty(B, dtype=torch.uint8, pin_memory=True)
    np_in, np_out, np_conv = h_in.numpy(), h_out.numpy(), h_conv.numpy()

    def sync_all():
        for k in range(N):
            torch.cuda.synchronize(k)

    cnt = None
    for _ in range(max(args.warmup, 3)):
        cnt = dec.decode_raw(B, np_in, lib.FMT_BITS, 0, np_out, lib.FMT_BITS, 0, np_conv)
    sync_all()
    sampler = ClockSampler(0)
    sampler.start()
    l0 = dec.launch_count()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cnt = dec.decode_raw(B, np_in, lib.FMT_BITS, 0, np_out, lib.FMT_BITS, 0, np_conv)
    sync_all()
    dt = time.perf_counter() - t0
    clocks = sampler.stop()
    launches = dec.launch_count() - l0
    value = B * args.steps / dt
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": N, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "mode": "single-process: one ldpcb200 handle over %d devices" % N,
            "config": config_dict(args, H, per, mi, B, {"host_memory": "pinned", "format": "BitMatrix in / BitMatrix out"}),
            "mean_iters": float(cnt[2]) / max(float(cnt[0]), 1.0), "converged_frac": float(cnt[1]) / max(float(cnt[0]), 1.0),
            "counters_match_single_device_run": bool(int(cnt[0]) == int(want[0]) and int(cnt[1]) == int(want[1]) and int(cnt[2]) == int(want[2])),
            "converged_check": bool(int(np_conv.sum()) == int(want[1])),
            "counters_via_nccl": bool(info["counters_via_nccl"]),
            "gpu_launches": int(launches), "clocks": clocks,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": int(h_in.numel()), "d2h_bytes_per_step": int(nb_out + B),
                    "api": "ldpcb200_decode_batch on a %d-device handle (FMT_BITS in/out, pinned host buffers); `value` IS this end-to-end number: "
                           "the timed region is the blocking host call" % N},
            "roofline": None,
            "kernel": {k: info[k] for k in ("family", "kernel_mode", "ctas_per_sm", "threads_per_cta", "kernel_rev", "ndev")},
            "note": "wall clock around the blocking call on a fixed host batch; the device-resident weak-scaling figure is the default mode"}
    dec.close()
    emit(line)


if __name__ == "__main__":
    main()
