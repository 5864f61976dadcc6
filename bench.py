#!/usr/bin/env python
"""bench.py -- depth-maps/s of the PatchmatchNet cascade with the B200-native PatchMatch hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo (one JSON line on rank 0)
    python bench.py ... --dump-outputs DIR                          # also write the last timed step's outputs as .npy
    python bench.py --impl reference [--steps K] [--warmup W]      # the reference algorithm on the host CPU

Workload (BASELINE.json configs[1]): 1 reference + 4 source views, 640x512, full 3-stage cascade with
64/32 -> 16/16 -> 8 hypotheses, one reference view per GPU (weak scaling: N GPUs -> N depth maps per step,
no collective on the data path).  A "step" is one full forward over one batch of synthetic input.

Numbers on the JSON line
    value      depth-maps/s, inputs resident in HBM, forward replayed from a CUDA graph, L2 flushed
               between timed steps, device time by CUDA events, max over ranks
    e2e        same metric through the public API (DepthEngine.infer_stream): pinned HOST inputs copied
               to the device and results copied back inside the timed region, every step
    roofline   the dominant hand-written kernel (fused warp+correlation, all source views per launch):
               algorithmic bytes per launch / CUDA-event duration of that launch, against the measured
               HBM copy bandwidth in MEASURED_PEAKS.json
    cpu_baseline  the oracle (CPU restatement of the reference, bit-identical to it) timed on the host
    gpu_eager_reference  the same oracle in eager PyTorch on the GPU, issuing the reference's own op sequence
               (what the unmodified reference would do on this B200; SURVEY.md 8d "honest bar")
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import torch

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)


def _synthetic():
    """patchmatchnet_b200.synthetic, imported lazily: `--impl reference` sets PMB200_SKIP_TORCH_OPS first so that the
    reference process maps none of the repo's native libraries (VERDICT r1, weak 6e)."""
    from patchmatchnet_b200 import synthetic

    return synthetic


WEIGHTS = os.path.join(REPO, "tests", "golden", "weights_000007.pt")
METRIC = "depth-maps/sec (1ref+4src, 640x512)"
UNIT = "depth-maps/s"


def build_net(patchmatch_cls=None):
    from patchmatchnet_b200.net import PatchmatchNet, load_reference_state

    synthetic = _synthetic()
    kw = dict(synthetic.DEFAULT_NET_KWARGS)
    net = PatchmatchNet(**kw) if patchmatch_cls is None else PatchmatchNet(**kw, patchmatch_cls=patchmatch_cls)
    if os.path.exists(WEIGHTS):
        load_reference_state(net, torch.load(WEIGHTS, map_location="cpu"))
        weights = "reference checkpoint params_000007 (fixture)"
    else:  # random init; give the zero-initialised offset convs something to do
        g = torch.Generator().manual_seed(0)
        for m in (net.patchmatch_1, net.patchmatch_2, net.patchmatch_3):
            for conv in (m.propa_conv, m.eval_conv):
                conv.weight.data.normal_(0, 0.05, generator=g)
        weights = "random init"
    return net.eval(), weights


# ----------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region.

    The timed region of the default run is ~20 ms, far shorter than the start-up of an `nvidia-smi -lms` process, so the
    primary sampler is an NVML thread (pynvml / nvidia-ml-py: one clock + one reasons query every ~2 ms, GIL released
    inside the library calls); `nvidia-smi -lms 20`, started BEFORE the warm-up so that it is already printing, is the
    fallback when NVML cannot be loaded.  Only samples taken between mark_begin() and mark_end() are reported; when the
    window caught none (nvidia-smi fallback on a very short run) the samples of the warm-up just before it are used and
    the line says so."""

    Q = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    NAMES = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")

    def __init__(self, gpu_index: int, device_uuid: str = ""):
        self.gpu = gpu_index
        self.uuid = device_uuid
        self.proc = None
        self.path = None
        self.thread = None
        self.samples = []  # (perf_counter, sm_mhz, reasons tuple)   [NVML thread]
        self.max_mhz = None
        self._stop = False
        self.t_begin = self.t_end = None
        self.wall_begin = self.wall_end = None

    # ---- NVML thread -------------------------------------------------------------------------------------------
    def _nvml_handle(self):
        import pynvml

        pynvml.nvmlInit()
        if self.uuid:
            for cand in (self.uuid, "GPU-" + self.uuid):
                for arg in (cand, cand.encode()):  # str or bytes, depending on the nvidia-ml-py version
                    try:
                        return pynvml, pynvml.nvmlDeviceGetHandleByUUID(arg)
                    except Exception:  # noqa: BLE001
                        continue
        return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.gpu)

    def _run_nvml(self, nv, h):
        bits = ((nv.nvmlClocksEventReasonHwSlowdown, "hw_slowdown"), (nv.nvmlClocksEventReasonHwThermalSlowdown, "hw_thermal_slowdown"),
                (nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_thermal_slowdown"), (nv.nvmlClocksEventReasonSwPowerCap, "sw_power_cap"))
        while not self._stop:
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                self.samples.append((time.perf_counter(), mhz, tuple(n for b, n in bits if mask & b)))
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.002)

    def start(self):
        try:
            import threading

            nv, h = self._nvml_handle()
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._run_nvml, args=(nv, h), daemon=True)
            self.thread.start()
            return
        except Exception:  # noqa: BLE001
            self.thread = None
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.gpu)],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL,
            )
        except Exception:  # noqa: BLE001
            self.proc = None

    def mark_begin(self):
        self.t_begin, self.wall_begin = time.perf_counter(), time.time()

    def mark_end(self):
        self.t_end, self.wall_end = time.perf_counter(), time.time()

    # ---- results -----------------------------------------------------------------------------------------------
    @staticmethod
    def _summary(rows, max_mhz, how, window):
        """rows: (sm_mhz, reasons tuple)"""
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": max_mhz, "reasons": ["no samples"], "how": how}
        reasons = sorted({r for _, rs in rows for r in rs})
        return {"sm_mhz": statistics.median(m for m, _ in rows), "sm_max_mhz": max_mhz, "reasons": reasons, "samples": len(rows),
                "how": how, "window": window}

    def stop(self):
        if self.thread is not None:
            self._stop = True
            self.thread.join(timeout=2)
            lo = self.t_begin if self.t_begin is not None else -1.0
            hi = self.t_end if self.t_end is not None else float("inf")
            inside = [(m, r) for t, m, r in self.samples if lo <= t <= hi]
            if inside:
                return self._summary(inside, self.max_mhz, "NVML thread, 2 ms period", "timed region")
            return self._summary([(m, r) for _, m, r in self.samples], self.max_mhz, "NVML thread, 2 ms period", "warm-up + timed region")
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML and nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        rows, mx = [], []
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    stamp = time.mktime(time.strptime(f[0].split(".")[0], "%Y/%m/%d %H:%M:%S")) + float("0." + f[0].split(".")[1])
                    mhz = float(f[1])
                    mx.append(float(f[2]))
                except (ValueError, IndexError):
                    continue
                rows.append((stamp, mhz, tuple(nm for nm, val in zip(self.NAMES, f[5:9]) if val.lower().startswith("active"))))
        finally:
            try:
                os.unlink(self.path)
            except OSError:
                pass
        top = max(mx) if mx else None
        if self.wall_begin is not None and self.wall_end is not None:
            inside = [(m, r) for t, m, r in rows if self.wall_begin - 0.02 <= t <= self.wall_end + 0.02]
            if inside:
                return self._summary(inside, top, "nvidia-smi -lms 20", "timed region")
        return self._summary([(m, r) for _, m, r in rows], top, "nvidia-smi -lms 20", "warm-up + timed region")


# ----------------------------------------------------------------------------------------------
# CPU baseline (oracle port of the reference, host cores)
# ----------------------------------------------------------------------------------------------


def cpu_forward_timer(height: int, width: int, n_views: int):
    """The oracle port of the reference on the host CPU.  torch's default is one thread per core; on a
    many-core host the small ops of this network get SLOWER with every core added, so the thread count is
    calibrated first (one forward per candidate, ascending, stop when it stops paying) and the reference is
    given its best configuration."""
    from oracle.pm_oracle import PatchMatchOracle  # allowed here: cpu_baseline / --impl reference legs only

    cores = os.cpu_count() or 1
    net, _ = build_net(PatchMatchOracle)
    net.stack_views = False  # the reference runs FeatureNet view by view (net.py:203-208)
    inp = _synthetic().make_inputs(1, n_views, height, width, seed=0)

    def step():
        with torch.no_grad():
            t0 = time.perf_counter()
            net([i.clone() for i in inp["images"]], inp["intrinsics"].clone(), inp["extrinsics"].clone(), inp["depth_min"], inp["depth_max"])
            return time.perf_counter() - t0

    cands = sorted({c for c in (8, 16, 32, 64, cores) if c <= cores})
    best_t, best_c, tried = None, cands[0], {}
    for c in cands:
        torch.set_num_threads(c)
        step()  # warm-up at this thread count
        t = step()
        tried[c] = round(t, 3)
        if best_t is None or t < best_t:
            best_t, best_c = t, c
        elif t > 1.5 * best_t:
            break
    torch.set_num_threads(best_c)
    step.calibration = tried
    return step, best_c


def gpu_eager_reference(height: int, width: int, n_views: int, device, warmup: int = 3, iters: int = 10):
    """The reference's algorithm as the reference would run it on THIS GPU: the oracle port (bit-identical to the
    reference on CPU) in eager PyTorch, the caller-side shell issuing the reference's own op sequence (conv, BatchNorm,
    ReLU separately, view by view; no folding, no stacking), cudnn.benchmark on as in eval.py:301, the TF32 switch as the
    caller left it (bench.py's default: off, i.e. the library convolutions in fp32 -- the configuration whose depth maps
    match the timed ones).  A reported baseline (SURVEY.md 8d "honest bar"), never part of the product path."""
    from oracle.pm_oracle import PatchMatchOracle  # allowed here: baseline legs only
    import patchmatchnet_b200.net as net_mod

    net, _ = build_net(PatchMatchOracle)
    net = net.to(device).eval()
    net.stack_views = False
    inp = _synthetic().make_inputs(1, n_views, height, width, seed=0)
    imgs = [i.to(device) for i in inp["images"]]
    K, E = inp["intrinsics"].to(device), inp["extrinsics"].to(device)
    dmin, dmax = inp["depth_min"].to(device), inp["depth_max"].to(device)
    net_mod.LIBRARY_FAST_PATH = False
    try:
        with torch.no_grad():
            for _ in range(warmup):
                net([i.clone() for i in imgs], K.clone(), E.clone(), dmin, dmax)
            torch.cuda.synchronize(device)
            t0 = time.perf_counter()
            for _ in range(iters):
                net([i.clone() for i in imgs], K.clone(), E.clone(), dmin, dmax)
            torch.cuda.synchronize(device)
            dt = time.perf_counter() - t0
    finally:
        net_mod.LIBRARY_FAST_PATH = True
    return {"value": iters / dt, "unit": UNIT, "ms_per_step": 1e3 * dt / iters, "kind": "port",
            "how": f"oracle port of the reference in eager PyTorch on the same GPU, reference op sequence, inputs resident, "
                   f"{warmup} warm-up + {iters} timed forwards, synchronize-bracketed wall clock, cudnn.benchmark=True, "
                   f"cudnn.allow_tf32={torch.backends.cudnn.allow_tf32}"}


def run_reference_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    os.environ["PMB200_SKIP_TORCH_OPS"] = "1"  # this process must not map libpmb200*.so (nothing here calls them)
    step, cores = cpu_forward_timer(args.height, args.width, args.views)
    for _ in range(args.warmup):
        step()
    times = [step() for _ in range(args.steps)]
    total = sum(times)
    value = args.steps / total
    sample = (f"{args.steps} full forwards of the workload (1 depth map each) after {args.warmup} warm-up, {cores} torch threads "
              f"(best of calibration {step.calibration}, host has {os.cpu_count()} cores)")
    line = {
        "impl": "reference",
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_label(1, args.views, args.height, args.width),
                   "where": "host CPU, one process on rank 0 whatever --gpus says: for N GPUs compare against N x this value",
                   "weights": "reference checkpoint params_000007 (fixture)" if os.path.exists(WEIGHTS) else "random init"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# this repo
# ----------------------------------------------------------------------------------------------


class LaunchCounter:
    """Counts native (libpmb200.so) kernel launches issued through patchmatchnet_b200.ops."""

    NAMES = ("relative_projection", "pack_nhwc", "warp_corr", "aggregate_views", "offset_corr", "init_propagate", "adaptive_eval",
             "warp_corr_score", "warp_corr_view_weights", "offset_corr_weight", "aggregate_views_score",
             "conv2d_nhwc", "conv2d_tc5", "conv2d_tc5h", "conv_stem", "refine_low", "refine_full", "upsample2x_add_nhwc",
             "photometric_confidence")

    def __init__(self):
        from patchmatchnet_b200 import _native

        self.n = 0
        self.by_name = {}
        self._lib = _native.lib()
        self._orig = {}

    def __enter__(self):
        for nm in self.NAMES:
            fn = getattr(self._lib, "pmb200_" + nm)
            self._orig[nm] = fn

            def wrapped(*a, _fn=fn, _nm=nm):
                self.n += 1
                self.by_name[_nm] = self.by_name.get(_nm, 0) + 1
                return _fn(*a)

            setattr(self._lib, "pmb200_" + nm, wrapped)
        return self

    def __exit__(self, *exc):
        for nm, fn in self._orig.items():
            setattr(self._lib, "pmb200_" + nm, fn)


def warp_corr_algorithmic_bytes(V, B, C, G, H, W, D):
    """SURVEY.md 8(d): per source view 4*B*H*W*(2C + D + G*D) bytes; one launch processes V views."""
    return V * 4 * B * H * W * (2 * C + D + G * D)


def warp_corr_minimum_bytes(V, B, C, G, H, W, D):
    """What the fused launch must actually move: ref once, V source maps, depth, V weights, one output."""
    return 4 * B * H * W * (C * (1 + V) + D + V + G * D)


KA_ENTRIES = ("warp_corr", "warp_corr_score", "warp_corr_view_weights")


def _ka_row(n, a, k, times_s, peak_gbs):
    ref, src, depth, G = a[0], a[1], a[3], a[4]
    B, H, W, C = ref.shape
    V, D = src.shape[0], depth.shape[1]
    # An event pair also times a host stall when the GPU runs dry between the two records (a Python GC pause or a scheduler
    # hiccup longer than the parking sleep: run 17 had one 60 ms sample among 20 of 48 us).  Such samples measure the host, not
    # the kernel: anything above 5x the median is dropped and counted in the row.
    med = statistics.median(times_s)
    kept = [x for x in times_s if x <= 5.0 * med]
    dropped = len(times_s) - len(kept)
    times_s = kept
    t = statistics.mean(times_s)
    alg = warp_corr_algorithmic_bytes(V, B, C, G, H, W, D)
    per_view_out = n == "warp_corr" and (len(a) < 6 or a[5] is None) and k.get("view_weights") is None
    keeps_sims = n == "warp_corr_view_weights" and (k.get("keep_sims") or (len(a) > 6 and a[6]))
    out_floats = {"warp_corr": G * D * (V if per_view_out else 1), "warp_corr_score": D,
                  "warp_corr_view_weights": V + (G * D * V if keeps_sims else 0)}[n]
    return {"entry": n, "shape": f"C{C} G{G} D{D} {H}x{W} V{V} B{B}", "us": 1e6 * t, "us_min": 1e6 * min(times_s),
            "algorithmic_bytes": alg, "minimum_bytes": 4 * B * H * W * (C * (1 + V) + D + V + out_floats),
            "achieved_gbs": alg / t / 1e9, "frac": alg / t / 1e9 / peak_gbs, "samples": len(times_s), "dropped_host_stall_samples": dropped}


def time_warp_corr_in_step(net, dev_inputs, peak_gbs, flush, steps=10, warmup=3):
    """Launch durations of the fused warp+correlation kernel measured LIVE inside timed steps: eager forwards
    (no graph, so events can bracket a launch), L2 flushed between steps -- not between kernels, the producer
    kernels of the same step leave their outputs in L2 exactly as in production -- one CUDA-event pair per K-A
    launch on the launching stream.  Covers warp_corr / warp_corr_score / warp_corr_view_weights."""
    from patchmatchnet_b200 import ops

    origs = {n: getattr(ops, n) for n in KA_ENTRIES}
    record = []  # (name, args, kwargs, start_event, end_event) per launch of the current step

    def make_spy(n):
        def spy(*a, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = origs[n](*a, **k)
            e1.record()
            record.append((n, a, k, e0, e1))
            return out
        return spy

    for n in KA_ENTRIES:
        setattr(ops, n, make_spy(n))
    per_call = []
    try:
        with torch.no_grad():
            for it in range(warmup + steps):
                record.clear()
                flush()
                # eager Python enqueues slower than the GPU drains (an eager forward is ~90 launches through Python, a few
                # ms of host time, for < 1.5 ms of device time): park the GPU (~30 ms) so the whole step is queued before
                # it starts, otherwise an event pair would also time the host's enqueue latency
                torch.cuda._sleep(60_000_000)
                torch.manual_seed(0)
                net(*dev_inputs())
                torch.cuda.synchronize()
                if it >= warmup:
                    for i, (n, a, k, e0, e1) in enumerate(record):
                        if len(per_call) <= i:
                            per_call.append((n, a, k, []))
                        per_call[i][3].append(e0.elapsed_time(e1) * 1e-3)
    finally:
        for n in KA_ENTRIES:
            setattr(ops, n, origs[n])
    return [_ka_row(n, a, k, ts, peak_gbs) for (n, a, k, ts) in per_call]


def time_eval_propagate_in_step(net, dev_inputs, peak_gbs, flush, steps=10, warmup=2):
    """K-B (adaptive evaluation) and K-C (initialisation / propagation) launches timed live inside eager steps, like K-A's:
    one row per launch of a step with SURVEY.md 8(d)'s algorithmic bytes -- K-B 4*B*H*W*(3D + 3K + 1), K-C 4*B*H*W*(Ns + 2Kp + (Ns + Kp)).
    Best effort: any surprise returns None and leaves the bench line as it is."""
    import inspect

    from patchmatchnet_b200 import ops

    names = ("adaptive_eval", "init_propagate")
    origs = {n: getattr(ops, n) for n in names}
    sigs = {n: inspect.signature(origs[n]) for n in names}
    record = []

    def make_spy(n):
        def spy(*a, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = origs[n](*a, **k)
            e1.record()
            try:
                b = sigs[n].bind(*a, **k).arguments
                if n == "adaptive_eval":
                    B, D, H, W = b["depth_sample"].shape
                    K = b["offsets"].shape[1] // 2
                    shape, alg = f"D{D} K{K} {H}x{W} B{B}", 4 * B * H * W * (3 * D + 3 * K + 1)
                else:
                    seed = b["seed_map"]
                    B, H, W = seed.shape[0], seed.shape[-2], seed.shape[-1]
                    Ns, Kp = int(b["Ns"]), int(b["Kp"])
                    shape, alg = f"Ns{Ns} Kp{Kp} {H}x{W} B{B}", 4 * B * H * W * (Ns + 2 * Kp + (Ns + Kp))
                record.append((n, shape, alg, e0, e1))
            except Exception:  # noqa: BLE001
                pass
            return out
        return spy

    per_call = []
    try:
        for n in names:
            setattr(ops, n, make_spy(n))
        with torch.no_grad():
            for it in range(warmup + steps):
                record.clear()
                flush()
                torch.cuda._sleep(60_000_000)  # park the GPU so that the whole step is queued before it starts (see K-A's)
                torch.manual_seed(0)
                net(*dev_inputs())
                torch.cuda.synchronize()
                if it >= warmup:
                    for i, (n, shape, alg, e0, e1) in enumerate(record):
                        if len(per_call) <= i:
                            per_call.append((n, shape, alg, []))
                        per_call[i][3].append(e0.elapsed_time(e1) * 1e-3)
    except Exception:  # noqa: BLE001
        return None
    finally:
        for n in names:
            setattr(ops, n, origs[n])
    rows = []
    for n, shape, alg, ts in per_call:
        med = statistics.median(ts)
        kept = [x for x in ts if x <= 5.0 * med] or ts
        t = statistics.mean(kept)
        rows.append({"entry": n, "kernel": "K-B" if n == "adaptive_eval" else "K-C", "shape": shape, "us": 1e6 * t, "us_min": 1e6 * min(kept),
                     "algorithmic_bytes": alg, "achieved_gbs": alg / t / 1e9, "frac": alg / t / 1e9 / peak_gbs,
                     "samples": len(kept), "dropped_host_stall_samples": len(ts) - len(kept)})
    return rows or None


def time_warp_corr_isolated(net, dev_inputs, peak_gbs, flush, iters=10):
    """The same launches re-run one at a time with L2 flushed before EACH launch (cold inputs from HBM)."""
    from patchmatchnet_b200 import ops

    calls = []
    origs = {n: getattr(ops, n) for n in KA_ENTRIES}

    def make_spy(n):
        def spy(*a, **k):
            calls.append((n, a, k))
            return origs[n](*a, **k)
        return spy

    for n in KA_ENTRIES:
        setattr(ops, n, make_spy(n))
    try:
        with torch.no_grad():
            torch.manual_seed(0)
            net(*dev_inputs())
    finally:
        for n in KA_ENTRIES:
            setattr(ops, n, origs[n])
    torch.cuda.synchronize()
    rows = []
    for (n, a, k) in calls:
        fn = origs[n]
        for _ in range(2):
            fn(*a, **k)
        ts = []
        for _ in range(iters):
            flush()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn(*a, **k)
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e-3)
        rows.append(_ka_row(n, a, k, ts, peak_gbs))
    return rows


def _recorded(stream):
    ev = torch.cuda.Event()
    ev.record(stream)
    return ev


def workload_label(B, N, H, W) -> str:
    base = f"1ref+{N - 1}src {W}x{H} 3-stage cascade (64/32,16/16,8 hyp), batch {B} per GPU"
    if (N, H, W) == (5, 512, 640):
        tag = "BASELINE.json configs[1]" if B == 1 else f"BASELINE.json configs[3]'s reference views, {B} on one GPU"
    elif (N, H, W) == (5, 1184, 1600) and B == 1:
        tag = "BASELINE.json configs[2]"
    else:
        tag = "custom size"
    return f"{base} ({tag})"


def bind_to_gpu_numa_node(local_rank: int) -> dict:
    """Pin this process (and therefore its pinned-host allocations, first-touch) to the CPUs NVML reports as local to the
    rank's GPU.  SCALE_r01: e2e efficiency at 8 GPUs was 0.93 with eight unbound processes pushing pinned H2D copies across
    both NUMA nodes.  Best effort: returns what it did for the JSON line."""
    try:
        import pynvml

        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = local_rank
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if local_rank < len(ids) and ids[local_rank].isdigit():
                idx = int(ids[local_rank])
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [w * 64 + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1 and w * 64 + b < ncpu]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return {"bound": False, "why": "NVML affinity set is empty or outside this process's cpuset"}
        os.sched_setaffinity(0, allowed)
        return {"bound": True, "cpus": f"{allowed[0]}-{allowed[-1]} ({len(allowed)})", "how": "nvmlDeviceGetCpuAffinity -> sched_setaffinity before pinned allocations"}
    except Exception as e:  # noqa: BLE001
        return {"bound": False, "why": repr(e)[:120]}


class Workload:
    """One (batch, views, size) problem on this rank: engine, resident device inputs, pinned host inputs."""

    def __init__(self, net, B, N, H, W, dev, slots, rank, use_graph=True):
        from patchmatchnet_b200.engine import DepthEngine

        synthetic = _synthetic()
        self.shape = (B, N, H, W)
        self.eng = DepthEngine(net, B, N, H, W, device=str(dev), use_graph=use_graph, n_slots=slots)
        host = synthetic.make_inputs(B, N, H, W, seed=rank)
        views = torch.stack(host["images"]).pin_memory()  # the request's views as adjacent slices of ONE pinned buffer: one upload
        self.host_pinned = dict(
            images=[views[i] for i in range(views.shape[0])],
            intrinsics=host["intrinsics"].pin_memory(), extrinsics=host["extrinsics"].pin_memory(),
            depth_min=host["depth_min"].pin_memory(), depth_max=host["depth_max"].pin_memory(),
        )
        self.d_in = dict(images=[im.to(dev) for im in host["images"]], intrinsics=host["intrinsics"].to(dev),
                         extrinsics=host["extrinsics"].to(dev), depth_min=host["depth_min"].to(dev), depth_max=host["depth_max"].to(dev))
        for s in range(self.eng.n_slots):
            self.eng.set_device_inputs(s, self.d_in["images"], self.d_in["intrinsics"], self.d_in["extrinsics"],
                                       self.d_in["depth_min"], self.d_in["depth_max"])
        torch.cuda.synchronize()

    def dev_inputs(self):
        d = self.d_in
        return ([im.clone() for im in d["images"]], d["intrinsics"].clone(), d["extrinsics"].clone(), d["depth_min"], d["depth_max"])


def time_resident(wl, steps, flush, stream, barrier):
    """K steps with inputs resident in HBM: rounds of up to `slots` concurrent graph replays, L2 flushed before every
    round outside the event pair that times it.  Returns the summed device seconds; `wl.last_step` is left holding the
    (depth, confidence) of the last step."""
    eng = wl.eng
    S = eng.n_slots
    rounds = [min(S, steps - r) for r in range(0, steps, S)]
    barrier()
    starts = [torch.cuda.Event(enable_timing=True) for _ in rounds]
    ends = [torch.cuda.Event(enable_timing=True) for _ in rounds]
    for i, n_now in enumerate(rounds):
        flush()
        starts[i].record(stream)
        wl.last_step = eng.run_round(n_now, starts[i], ends[i])[-1]
    barrier()
    return sum(s.elapsed_time(e) for s, e in zip(starts, ends)) * 1e-3


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy in float32.  When together they exceed DUMP_BYTES, each is replaced by
    the same fixed, seeded sample of its flattened elements (a share of the budget proportional to its size), so
    that two runs with the same arguments stay comparable element for element.  Returns what was written."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.numel() for a in arrays.values()) * 4
    written = {}
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        entry = {"shape": list(a.shape), "dtype": "float32"}
        if total > DUMP_BYTES:
            keep = max(1, a.size * DUMP_BYTES // total)
            idx = np.sort(np.random.default_rng(0).choice(a.size, size=keep, replace=False))
            a = a.reshape(-1)[idx]
            entry["sample"] = f"{keep} of {t.numel()} elements, flat indices np.random.default_rng(0).choice({t.numel()}, {keep}, replace=False), sorted"
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a, dtype=np.float32))
        written[name] = entry
    return written


def time_e2e(wl, steps, stream, barrier):
    """K requests through the public API: pinned host in -> device -> graph -> pinned host out, every request."""
    eng = wl.eng
    reqs = [wl.host_pinned] * steps
    barrier()
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record(stream)
    eng.copy_stream.wait_event(t0)
    for sl in eng._slots:
        sl["stream"].wait_event(t0)
    h2d, d2h = eng.infer_stream(reqs)  # returns after every slot stream has drained
    t1.record(stream)
    barrier()
    return t0.elapsed_time(t1) * 1e-3, h2d, d2h


def single_request_latency(wl, flush, stream, iters=10):
    """One request alone on the GPU: device time of one graph replay (inputs resident, L2 flushed) and the wall-clock of
    the synchronous public call (pinned host in -> pinned host out)."""
    eng = wl.eng
    dev_ms, wall_ms = [], []
    for _ in range(iters):
        flush()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        eng.run_slot(0)
        e1.record(stream)
        e1.synchronize()
        dev_ms.append(e0.elapsed_time(e1))
    h = wl.host_pinned
    for _ in range(iters):
        t0 = time.perf_counter()
        eng.infer(h["images"], h["intrinsics"], h["extrinsics"], h["depth_min"], h["depth_max"])
        wall_ms.append(1e3 * (time.perf_counter() - t0))
    return {"device_ms": statistics.median(dev_ms), "device_ms_min": min(dev_ms), "host_to_host_ms": statistics.median(wall_ms),
            "how": f"median of {iters}: one CUDA-graph replay alone on the GPU, L2 flushed, CUDA events; and DepthEngine.infer wall clock"}


def ka_roofline(net, wl, peak_gbs, peak_src, flush, steps):
    detail = time_warp_corr_in_step(net, wl.dev_inputs, peak_gbs, flush, steps=steps)
    if not detail:
        return None, detail
    n_l = len(detail)
    alg_mean = sum(r["algorithmic_bytes"] for r in detail) / n_l
    us_mean = sum(r["us"] for r in detail) / n_l
    traffic, traffic_src = None, None
    tfile = os.path.join(REPO, "profiles", TRAFFIC_FILE)
    if os.path.exists(tfile):
        try:
            t = json.load(open(tfile))
            traffic, traffic_src = t.get("mean_dram_bytes_per_launch"), f"profiles/{TRAFFIC_FILE} ({t.get('capture', 'ncu --set full')})"
        except Exception:  # noqa: BLE001
            traffic = None
    achieved = alg_mean / (us_mean * 1e-6) / 1e9
    roofline = {"bound": "hbm", "kernel": f"fused warp + bilinear gather + group correlation + view aggregation + head (K-A), {n_l} launches per step",
                "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs, "traffic": traffic,
                "traffic_source": traffic_src,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_mean, "us_per_launch": us_mean,
                "how": "mean over the kernel's launches of one step; each launch timed by a CUDA-event pair inside timed eager steps "
                       "(L2 flushed between steps, GPU parked so the host's enqueue latency is not measured); "
                       "algorithmic bytes = V * 4*B*H*W*(2C + D + G*D) per launch (SURVEY.md 8d)",
                "best_launch_frac": max(r["frac"] for r in detail), "worst_launch_frac": min(r["frac"] for r in detail)}
    return roofline, detail


TRAFFIC_FILE = "r2_warp_corr_traffic.json"  # written from this round's ncu --set full capture (tools/summarize_ncu.py)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--height", type=int, default=512)
    ap.add_argument("--width", type=int, default=640)
    ap.add_argument("--views", type=int, default=5, help="1 reference + (views-1) sources")
    ap.add_argument("--batch", type=int, default=1, help="reference views per GPU")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="skip the eager-PyTorch reference timing on the GPU")
    ap.add_argument("--tf32", action="store_true", help="time torch's default flags instead (TF32 operands in the convolutions): faster, but the "
                    "depth maps are 2.6e-3..3.3e-3 off the fp32 reference, outside north_star's 1e-3 (tests/test_gpu_bench_mode.py)")
    ap.add_argument("--no-tf32", action="store_true", help="accepted for compatibility: fp32-accurate convolutions are the default")
    ap.add_argument("--slots", type=int, default=3, help="independent requests in flight per GPU (each its own stream + CUDA graph)")
    ap.add_argument("--cpu-samples", type=int, default=4)
    ap.add_argument("--repeats", type=int, default=5, help="the K-step timed region is repeated this many times; the line reports the median")
    ap.add_argument("--no-sub", action="store_true", help="skip the fp32 / 1600x1184 / batch-8 sub-records (N=1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the depth map and confidence of the last timed step as DIR/<name>.npy "
                         "(float32; rank 0; a fixed seeded sample when they exceed 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        run_reference_arm(args)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    numa = bind_to_gpu_numa_node(local)  # before any pinned allocation
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    torch.backends.cudnn.benchmark = True  # as the reference's eval.py:301 does; autotuned during warm-up
    # Default: every convolution fp32-accurate (native 3xTF32 split on the tensor cores) -- the configuration the parity tests
    # hold to north_star's 1e-3 (observed ~1e-5).  --tf32 leaves torch's default (TF32 operands).
    args.no_tf32 = not args.tf32
    if args.no_tf32:
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist_mod.init_process_group("nccl", device_id=dev)
        dist = dist_mod

    B, N, H, W = args.batch, args.views, args.height, args.width
    torch.manual_seed(0)  # the random depth hypotheses stage 3 draws on the GPU: the same arguments, the same outputs
    net, weights = build_net()
    wl = Workload(net, B, N, H, W, dev, args.slots, rank, use_graph=not args.no_graph)
    eng = wl.eng

    with LaunchCounter() as lc:
        eng.prepare()  # warm-up forwards + graph capture
    forwards_counted = eng.n_slots * (eng._warmup + (1 if eng.use_graph else 0))
    launches_per_step = lc.n // max(1, forwards_counted)

    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def flush():
        flush_buf.zero_()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(vals):
        if dist is None:
            return list(vals)
        t = torch.tensor(list(vals), device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    # ---------------- kernel-side throughput: inputs resident in HBM ----------------
    stream = torch.cuda.current_stream()
    S = eng.n_slots
    try:
        uuid = str(torch.cuda.get_device_properties(dev).uuid)
    except Exception:  # noqa: BLE001
        uuid = ""
    sampler = ClockSampler(local, uuid)
    sampler.start()  # before the warm-up: the sampler is already running when the timed region starts
    for _ in range(max(1, (args.warmup + S - 1) // S)):
        flush()
        eng.run_round(S, _recorded(stream), torch.cuda.Event())
    barrier()
    sampler.mark_begin()
    dev_runs = [time_resident(wl, args.steps, flush, stream, barrier) for _ in range(max(1, args.repeats))]
    sampler.mark_end()
    last_step = {"depth": wl.last_step[0].cpu(), "confidence": wl.last_step[1].cpu()}  # before later phases reuse the slots
    clocks = sampler.stop()
    dev_runs = reduce_max(dev_runs)  # per repeat: the slowest rank
    dev_seconds = statistics.median(dev_runs)

    # ---------------- end to end: pinned host in, pinned host out, every step ----------------
    eng.infer_stream([wl.host_pinned] * max(args.warmup, eng.n_slots))
    e2e_runs, h2d, d2h = [], 0, 0
    for _ in range(max(1, args.repeats)):
        t, h2d, d2h = time_e2e(wl, args.steps, stream, barrier)
        e2e_runs.append(t)
    e2e_runs = reduce_max(e2e_runs)
    e2e_seconds = statistics.median(e2e_runs)

    maps = args.steps * B * world
    value = maps / dev_seconds
    e2e_value = maps / e2e_seconds

    # ---------------- roofline of the dominant kernel + baselines + sub-records (rank 0) ----------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    roofline, detail, detail_cold, cpu_baseline, gpu_eager, latency, sub = None, None, None, None, None, None, {}
    detail_kb_kc = None
    if rank == 0:
        roofline, detail = ka_roofline(net, wl, peak_gbs, peak_src, flush, steps=max(5, args.steps // 2))
        detail_cold = time_warp_corr_isolated(net, wl.dev_inputs, peak_gbs, flush)
        try:
            detail_kb_kc = time_eval_propagate_in_step(net, wl.dev_inputs, peak_gbs, flush, steps=max(5, args.steps // 2))
        except Exception:  # noqa: BLE001
            detail_kb_kc = None
        latency = single_request_latency(wl, flush, stream)
    if world == 1 and not args.no_sub:
        # (1) the same workload under torch's default flags (TF32 operands in the convs), as round 1 timed it: own net so that
        #     the precision-keyed weight caches captured by the graphs above are not evicted.  Reported, not the headline:
        #     its depth maps are outside the 1e-3 parity bound.
        if args.no_tf32:
            old = torch.backends.cudnn.allow_tf32
            torch.backends.cudnn.allow_tf32 = True
            try:
                net_t, _ = build_net()
                wl_t = Workload(net_t, B, N, H, W, dev, args.slots, rank, use_graph=not args.no_graph)
                wl_t.eng.prepare()
                runs = [time_resident(wl_t, args.steps, flush, stream, barrier) for _ in range(3)]
                sub["value_tf32"] = {"value": args.steps * B / statistics.median(runs), "unit": UNIT,
                                     "ms_per_step": 1e3 * statistics.median(runs) / args.steps,
                                     "parity": "OUTSIDE the bound: depth rel-L1 vs the fp32 oracle 2.6e-3 (cfg 2) / 3.3e-3 (cfg 3) / 3.1e-3 (B=8), "
                                               "north_star allows 1e-3 (tests/test_gpu_bench_mode.py, profiles/r2_run1_bench_mode_parity.json)",
                                     "how": "same workload, torch default cudnn.allow_tf32=True: native convs with TF32 operands on the memory-bound "
                                            "layers, cuDNN TF32 on the FLOP-bound ones; median of 3"}
                del wl_t, net_t
            finally:
                torch.backends.cudnn.allow_tf32 = old
        # (2) BASELINE config 3 (DTU full size) and 8 reference views on one GPU: value, e2e and the K-A roofline there
        for key, (b2, h2, w2, s2, st2) in {"cfg3_1600x1184": (1, 1184, 1600, 2, 10), "batch8_640x512": (8, 512, 640, 1, 5)}.items():
            if (b2, h2, w2) == (B, H, W):
                continue
            try:
                w2l = Workload(net, b2, N, h2, w2, dev, s2, rank, use_graph=not args.no_graph)
                w2l.eng.prepare()
                for _ in range(2):
                    time_resident(w2l, s2, flush, stream, barrier)
                runs = [time_resident(w2l, st2, flush, stream, barrier) for _ in range(3)]
                w2l.eng.infer_stream([w2l.host_pinned] * max(3, s2))
                e_runs = [time_e2e(w2l, st2, stream, barrier)[0] for _ in range(3)]
                rl, det = ka_roofline(net, w2l, peak_gbs, peak_src, flush, steps=5)
                sub[key] = {"workload": workload_label(b2, N, h2, w2), "value": st2 * b2 / statistics.median(runs), "unit": UNIT,
                            "ms_per_step": 1e3 * statistics.median(runs) / st2, "e2e_value": st2 * b2 / statistics.median(e_runs),
                            "requests_in_flight": s2, "steps": st2, "repeats": 3,
                            "roofline": None if rl is None else {k: rl[k] for k in ("achieved", "peak", "frac", "us_per_launch", "algorithmic_bytes_per_launch", "best_launch_frac", "worst_launch_frac")},
                            "roofline_detail": None if det is None else [{k: r[k] for k in ("shape", "us", "frac")} for r in det]}
                del w2l
                torch.cuda.empty_cache()
            except Exception as e:  # noqa: BLE001
                sub[key] = {"error": repr(e)[:300]}
    if rank == 0:
        if world == 1 and not args.no_gpu_baseline:
            gpu_eager = gpu_eager_reference(H, W, N, dev)
        if world == 1 and not args.no_cpu_baseline:
            step, cores = cpu_forward_timer(H, W, N)
            step()
            ts = [step() for _ in range(args.cpu_samples)]
            cpu_baseline = {"value": len(ts) / sum(ts), "unit": UNIT, "cores": cores, "kind": "port",
                            "sample": f"{len(ts)} full forwards of the same workload (after 1 warm-up) with the oracle port of the reference, "
                                      f"{cores} torch threads (best of calibration {step.calibration}, host has {os.cpu_count()} cores)"}

    if rank == 0:
        tf32 = not args.no_tf32
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dev_seconds / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 kernels + tf32-operand convs (torch default cudnn.allow_tf32; outside the 1e-3 parity bound)" if tf32
                     else "f32 (PatchMatch kernels fp32; every conv on the tensor cores with the error-compensated 3xTF32 split, fp32-accurate)",
            "data": "synthetic",
            "repeats": {"n": len(dev_runs), "statistic": "median", "value_min": maps / max(dev_runs), "value_max": maps / min(dev_runs),
                        "e2e_min": maps / max(e2e_runs), "e2e_max": maps / min(e2e_runs),
                        "ms_per_step_all": [round(1e3 * t / args.steps, 4) for t in dev_runs]},
            "config": {"workload": workload_label(B, N, H, W),
                       "parallelism": f"{world} x (1 process/GPU, reference views sharded by rank, no data-path collective)",
                       "weights": weights, "cuda_graph": eng.use_graph, "requests_in_flight": eng.n_slots,
                       "l2": "flushed before every timed round of <= requests_in_flight concurrent steps (256 MiB write, outside the events)",
                       "convs": ("every conv (FeatureNet, Refinement, offset convs) on the native channels-last tensor-core kernel, 3xTF32 "
                                 "error-compensated split = fp32-accurate; no cuDNN conv in the step. Parity of THIS mode: "
                                 "tests/test_gpu_bench_mode.py (depth rel-L1 vs the fp32 oracle ~1e-5)" if not tf32 else
                                 "native channels-last tensor-core convs (TF32 operands, fp32 accumulate) for FeatureNet's memory-bound layers, "
                                 "its top-down path, Refinement and the stage-1 offset conv; cuDNN (TF32 allowed, torch's default) for the "
                                 "FLOP-bound FeatureNet layers and the stage-2/3 offset convs; every PatchMatch kernel is full fp32. "
                                 "This mode is OUTSIDE the 1e-3 parity bound (tests/test_gpu_bench_mode.py)"),
                       "numa": numa},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": 1e3 * e2e_seconds / args.steps,
                    "how": "DepthEngine.infer_stream: pinned host inputs -> device (copy stream) -> CUDA graph on the request's slot stream -> pinned host outputs; "
                           "requests_in_flight independent requests overlap"},
            "latency_single_request": latency,
            "gpu_launches": launches_per_step * args.steps, "gpu_launches_per_step": launches_per_step,
            "native_kernels_per_step": {k: v // max(1, forwards_counted) for k, v in sorted(lc.by_name.items())},
            "clocks": clocks,
            "roofline": roofline, "roofline_detail": detail, "roofline_detail_cold_isolated": detail_cold,
            "roofline_detail_eval_propagate": detail_kb_kc,
            "cpu_baseline": cpu_baseline,
            "gpu_eager_reference": gpu_eager,
        }
        line.update(sub)
        if args.dump_outputs:
            line["dumped_outputs"] = {"dir": args.dump_outputs, "step": "last timed step of the last repeat",
                                      "arrays": dump_outputs(args.dump_outputs, last_step)}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
