#!/usr/bin/env python
"""Benchmark of the plane-sweep cost-volume hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload cfg2|cfg1|cfg3|cfg4|stress_dot|stress_hero] [--no-also] [--dump-outputs DIR]

A *step* is one pass of the hot path over one batch of synthetic frame tuples: one
``FeatureVolumeManager.forward`` (hero, metadata-MLP matching) or ``CostVolumeManager.forward``
(dot) call.  The DEFAULT workload is the hero model at 8 frames per GPU, 1 ref + 7 source
views, 640x480 frames -> 120x160 matching maps, D = 64: at N = 1 that is BASELINE.json
``configs[2]`` (batch 8 on one B200) and at N = 8 it is ``configs[4]`` (batch 64 over 8 GPUs, the
1/2/4/8 scaling curve).  The dot-product configuration the metric was first quoted on
(``configs[1]``, batch 4) is measured in the same run and reported under ``"also"``.
With N GPUs every rank processes its own batch (frames are independent: weak scaling, no
data-path collective); NCCL is used for the barrier and the MAX-reduce of the elapsed time.

Prints ONE JSON line (rank 0).  Keys beyond the base contract:
  roofline      hero: bound "tensor" — algorithmic MLP FLOPs per sweep launch / measured launch
                time against MEASURED_PEAKS.json bf16_tflops_sustained (the kernel is timed inside
                a long loop); `issued_mma` = the same with the three fp16 MMAs per product the
                hi/lo split issues; `hbm` = the algorithmic-bytes fraction the metric asks for.
                dot: bound "hbm" + `binding` (the on-chip gather path that actually bounds it,
                against the MEASURED L1 ceiling of scripts/probes/l1_gather_probe).
                `traffic` = ncu dram bytes per launch cited from profiles/ (`traffic_source`).
  cpu_baseline  the oracle's reference-structured port (oracle/costvolume_oracle.py,
                sampler="aten": the reference's op sequence) timed on the host cores
  e2e           same metric through the public manager API with HOST (pinned) inputs
                and outputs: H2D + sweep + D2H inside the timed region; median of 3 windows
`--impl reference` times the CPU port alone on the SAME config (the reference is pure
Python/PyTorch and not part of this repository; the port is op-for-op the reference's own sequence
and is pinned against its recorded outputs in tests/test_oracle_vs_reference.py);
each step is a bounded sample of the batch (stated in `cpu_baseline.sample`), the metric is per frame.
`--dump-outputs DIR` writes what the last timed step returned (rank 0) as DIR/<workload>_<output>.npy,
float32, so that two builds can be compared output for output: the inputs are seeded and depend only
on the arguments.  Past 64 MB in all, each array is replaced by a fixed seeded sample of its flattened
elements (the same sample for the same shape).
"""
from __future__ import annotations

import argparse
import contextlib
import json
import os
import statistics
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

METRIC = "cost_volume_frames_per_sec@640x480_D64_K7src"
UNIT = "frames/s"
L2_BYTES = 126 * 1024 * 1024
DUMP_BYTES = 64 * 10**6
OUTPUT_NAMES = ("cost_volume", "lowest_cost", "depth_planes", "overall_mask")
DEFAULT_WORKLOAD = "cfg2"
ALSO_WORKLOAD = "cfg1"
# frames per GPU (weak scaling): the single-GPU configuration's batch
PER_GPU = {"cfg0": 1, "cfg1": 4, "cfg2": 8, "cfg3": 4, "cfg4": 8}
# measured by scripts/probes/l1_gather_probe on a B200 (profiles/r02_l1_gather_probe.jsonl):
# bytes the LSU/L1 path delivers to the dot sweep's exact load shape (warp-wide LDG.128 of
# 256-byte row segments) per clock and SM at 16 / 32 / 64 resident warps
L1_GATHER_B_PER_CLK_SM = {16: 127.6, 32: 145.0, 64: 194.4}


def algorithmic_bytes_per_frame(w, hero: bool, with_mask: bool) -> int:
    """SURVEY.md §8(d): compulsory HBM traffic of one reference frame."""
    HW = w.height * w.width
    b = 4 * (w.channels * HW + w.views * w.channels * HW + w.planes * HW + HW)
    b += 4 * (48 * w.views + 16) + 4 * w.planes
    if hero and with_mask:
        b += HW
    return b


def mlp_flops_per_frame(w, issued: bool) -> float:
    """SURVEY.md §8(d): 2 * D * HW * (F*128 + 128*128 + 128) algorithmic; `issued` counts what the
    tcgen05 kernel actually issues: layer-1 K = 192 (the 21 pose measures enter as a per-frame bias,
    182 live positions padded to 12 K-steps), three fp16 MMAs per product, layer 3 on SIMT."""
    rows = w.planes * w.height * w.width
    f_in = w.channels * (w.views + 1) + 10 * w.views + 4
    if issued:
        return 2.0 * 3 * rows * (192 * 128 + 128 * 128)
    return 2.0 * rows * (f_in * 128 + 128 * 128 + 128)


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.is_file():
        d = json.loads(p.read_text())
        return {"hbm_gbs": float(d["hbm_gbs"]), "tf_burst": float(d["bf16_tflops"]),
                "tf_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0,
            "source": "fallback (B200_PROFILING.md)"}


def load_traffic(tag: str):
    """dram bytes per launch of the dominant kernel, cited from a committed ncu summary."""
    p = ROOT / "profiles" / "ncu_traffic.json"
    if p.is_file():
        try:
            d = json.loads(p.read_text())
            return d.get(tag), d.get("_source", {}).get(tag, "profiles/ncu_traffic.json")
        except Exception:
            return None, None
    return None, None


def make_roofline(w, hero, frames, sweep_s, prep_s, step_s, variant, sm_mhz):
    pk = load_peaks()
    alg_bytes = algorithmic_bytes_per_frame(w, hero, True) * frames
    gbs = alg_bytes / sweep_s / 1e9
    traffic, tsrc = load_traffic(f"{w.kind}:{variant}")
    common = {
        "kernel": variant, "sweep_us_per_launch": sweep_s * 1e6, "prep_us_per_launch": prep_s * 1e6,
        "sweep_share_of_step": sweep_s / step_s, "peak_source": pk["source"],
        "traffic": traffic, "traffic_source": (f"cited from {tsrc} (one ncu --set full capture of this kernel at this "
                                               "batch; not re-measured by this run)") if traffic else None,
        "algorithmic_bytes_per_launch": alg_bytes,
    }
    hbm = {"achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"]}
    if hero:
        tf = mlp_flops_per_frame(w, False) * frames / sweep_s / 1e12
        tfi = mlp_flops_per_frame(w, True) * frames / sweep_s / 1e12
        return {
            "bound": "tensor", "achieved": tf, "peak": pk["tf_sustained"], "unit": "TFLOP/s",
            "frac": tf / pk["tf_sustained"],
            "peak_kind": "bf16_tflops_sustained (cuBLAS, seconds-long loop: this kernel is timed inside one)",
            "algorithmic_flops_per_launch": mlp_flops_per_frame(w, False) * frames,
            "issued_mma": {"achieved": tfi, "unit": "TFLOP/s", "frac_of_sustained": tfi / pk["tf_sustained"],
                           "frac_of_burst": tfi / pk["tf_burst"],
                           "what": "fp16 hi/lo split: 3 MMAs per product, layer-1 K = 192"},
            "hbm": hbm, **common,
            "note": ("the metadata-MLP sweep is a dense contraction at ~7000 FLOP/B: tensor-bound; the HBM "
                     "fraction the metric names is reported under `hbm`"),
        }
    sm = 148
    clk = (sm_mhz or 1965) * 1e6
    samples = frames * w.planes * w.views * w.height * w.width
    gather = samples * 4 * w.channels * 4
    ceil64 = L1_GATHER_B_PER_CLK_SM[64]
    return {
        "bound": "hbm", **hbm, **common,
        "binding": {"resource": "l1_gather_bytes", "achieved_B_per_clk_sm": gather / sweep_s / clk / sm,
                    "peak_B_per_clk_sm": ceil64, "frac": gather / sweep_s / clk / sm / ceil64,
                    "peak_source": ("measured: scripts/probes/l1_gather_probe, this load shape, 64 warps/SM "
                                    f"(16 warps: {L1_GATHER_B_PER_CLK_SM[16]}, 32: {L1_GATHER_B_PER_CLK_SM[32]}); "
                                    "profiles/r02_l1_gather_probe.jsonl"),
                    "sm_mhz_used": sm_mhz or 1965},
        "note": ("HBM fraction as the metric demands; at 116 FLOP/B the dot sweep is bound by the on-chip "
                 "gather path — see `binding` and DESIGN.md"),
    }


class ClockSampler:
    """Samples SM clock / throttle reasons through NVML while `active` is set."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.active = threading.Event()
        self._stop = threading.Event()
        self._ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self._ok = True
        except Exception:
            self._ok = False
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        if not self._ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop.is_set():
            if not self.active.is_set():
                time.sleep(0.0005)
                continue
            time.sleep(0.010)   # ~100 samples/s: NVML queries take driver locks that CUDA calls of the timed
                                # loop also need, and a busy poll would fight it for the GIL
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass

    def snapshot(self):
        if not self._ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}

    def reset(self):
        self.samples, self.reasons = [], set()

    def stop(self):
        self._stop.set()


# --------------------------------------------------------------------------- #
# CPU port (reference arm / cpu_baseline)                                     #
# --------------------------------------------------------------------------- #
def cpu_port_step(w, tup, weights):
    from oracle import costvolume_oracle as O
    if w.kind == "dot":
        return O.forward_dot(**tup, num_depth_bins=w.planes, sampler="aten")
    return O.forward_mlp(**tup, weights=weights, num_depth_bins=w.planes, return_mask=True,
                         sampler="aten")


def pick_cpu_threads(w) -> int:
    """The port is ATen ops on ~20 k-pixel tensors: on a many-core host more threads can be
    SLOWER (128 threads: 0.44 frames/s, 16 threads: >5 on the same box).  Probe a few thread
    counts on an 8-plane slice of one frame, twice each, and keep the fastest, so the baseline is the
    best the host can do, not an oversubscribed one.  $SRCV_CPU_THREADS fixes the count."""
    import dataclasses
    from oracle import costvolume_oracle as O
    from simplerecon_b200.synthetic import make_workload_tuple, mlp_state
    if os.environ.get("SRCV_CPU_THREADS"):
        n = int(os.environ["SRCV_CPU_THREADS"])
        torch.set_num_threads(n)
        return n
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cands = sorted({c for c in (8, 16, 32, 64, cores) if c <= cores})
    small = dataclasses.replace(w, planes=8)
    tup = make_workload_tuple(w, batch=1)
    weights = O.mlp_weights_from_state_dict(mlp_state(w.views, w.channels)) if w.kind == "mlp" else None
    best, best_t = cands[0], float("inf")
    with torch.inference_mode():
        for c in cands:
            torch.set_num_threads(c)
            cpu_port_step(small, tup, weights)
            dt = float("inf")
            for _ in range(2):
                t0 = time.perf_counter()
                cpu_port_step(small, tup, weights)
                dt = min(dt, time.perf_counter() - t0)
            if dt < 0.97 * best_t:          # a larger count must win clearly: keeps the choice stable
                best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def time_cpu_port(w, frames: int, min_seconds: float, max_reps: int):
    """Returns (frames_per_s, cores, sample description): mean over the timed repetitions."""
    from oracle import costvolume_oracle as O
    from simplerecon_b200.synthetic import make_workload_tuple, mlp_state
    cores = pick_cpu_threads(w)
    tup = make_workload_tuple(w, batch=frames)
    weights = O.mlp_weights_from_state_dict(mlp_state(w.views, w.channels)) if w.kind == "mlp" else None
    with torch.inference_mode():
        cpu_port_step(w, tup, weights)                       # warm-up
        reps, t_all = 0, time.perf_counter()
        while reps < max_reps and (time.perf_counter() - t_all < min_seconds or reps < 1):
            cpu_port_step(w, tup, weights)
            reps += 1
        dt = time.perf_counter() - t_all
    return frames * reps / dt, cores, (f"{frames} frame(s) of {w.name} per repetition, mean of {reps} after 1 "
                                       f"warm-up, {cores} of {os.cpu_count()} host threads (fastest of a probe)")


def time_c_port(w, frames: int):
    """The plain-C restatement (oracle/cv_oracle.c, OpenMP over pixels, all host threads): a CPU
    number that scales with the core count where the ATen-op port does not."""
    try:
        from oracle import c_oracle as CO
        from oracle import costvolume_oracle as O
        from simplerecon_b200.synthetic import make_workload_tuple, mlp_state
        tup = make_workload_tuple(w, batch=frames)
        if w.kind == "dot":
            fn = lambda: CO.forward_dot(**tup, num_depth_bins=w.planes)
        else:
            wts = O.mlp_weights_from_state_dict(mlp_state(w.views, w.channels))
            fn = lambda: CO.forward_mlp(**tup, weights=wts, num_depth_bins=w.planes, return_mask=True)
        fn()
        best = float("inf")
        for _ in range(2):
            t0 = time.perf_counter()
            fn()
            best = min(best, time.perf_counter() - t0)
        return {"value": frames / best, "unit": UNIT, "threads": os.cpu_count(),
                "sample": f"{frames} frame(s), best of 2, fp32 scalar loops + OpenMP"}
    except Exception as ex:  # pragma: no cover - informational only
        return {"value": None, "error": str(ex)[:200]}


def workload_config(w, batch_per_gpu, world):
    """Identical for the GPU arm and the reference arm (the driver compares them)."""
    in_bytes = 4 * batch_per_gpu * (w.channels * w.height * w.width * (1 + w.views))
    n_sets = max(2, -(-int(1.25 * L2_BYTES) // in_bytes))
    return {
        "workload": w.name, "matching": w.kind,
        "frame": "n/a (stress: feature map given directly)" if w.name.startswith("stress")
        else f"{4 * w.width}x{4 * w.height}",
        "feature_map": f"{w.width}x{w.height}", "planes": w.planes, "src_views": w.views,
        "channels": w.channels, "batch_per_gpu": batch_per_gpu, "global_batch": batch_per_gpu * world,
        "parallelism": f"frame-sharded x{world} (no data-path collective)",
        "l2": (f"{n_sets} rotating input sets, {n_sets * in_bytes / 2**20:.0f} MiB > 126 MiB L2; "
               f"outputs ({4 * batch_per_gpu * w.planes * w.height * w.width / 2**20:.0f} MiB/step) freshly allocated"),
    }, n_sets


def run_reference_arm(args, w, per_gpu):
    """`--impl reference`: the reference's CPU implementation (port) of the same workload and
    config, all the host threads it can use, rank 0 only.  Each step is a bounded sample of the
    batch (the metric is per frame), sized so that the whole run ends within a few minutes."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    from oracle import costvolume_oracle as O
    from simplerecon_b200.synthetic import make_workload_tuple, mlp_state
    cores = pick_cpu_threads(w)
    weights = O.mlp_weights_from_state_dict(mlp_state(w.views, w.channels)) if w.kind == "mlp" else None
    # size the per-step sample from one timed frame: the whole run should stay under ~150 s
    one = make_workload_tuple(w, batch=1)
    with torch.inference_mode():
        cpu_port_step(w, one, weights)
        t0 = time.perf_counter()
        cpu_port_step(w, one, weights)
        t_frame = time.perf_counter() - t0
    budget = float(os.environ.get("SRCV_REF_BUDGET_S", "150"))   # seconds for the whole run (tests shrink it)
    n_steps = args.steps + max(1, min(args.warmup, 2))
    share = budget / (t_frame * n_steps)            # frames per step the budget allows
    frames = int(max(1, min(per_gpu, share)))
    # Many steps (the no-flag default is 100): even one frame per step would take minutes, so a step
    # is then a plane subset of ONE frame — the port loops over planes like the reference
    # (modules/cost_volume.py:305, :557), every plane costs the same, the metric stays per frame.
    planes_timed = w.planes if share >= 1.0 else int(max(4, min(w.planes, w.planes * share)))
    import dataclasses
    w_timed = dataclasses.replace(w, planes=planes_timed)
    tup = make_workload_tuple(w, batch=frames)
    with torch.inference_mode():
        for _ in range(max(1, min(args.warmup, 2))):
            cpu_port_step(w_timed, tup, weights)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            cpu_port_step(w_timed, tup, weights)
        dt = time.perf_counter() - t0
    fps = frames * (planes_timed / w.planes) * args.steps / dt
    what = (f"{frames} of the {per_gpu} frames of a batch per step" if planes_timed == w.planes else
            f"{planes_timed} of the {w.planes} planes of one frame per step (the port's plane loop is uniform)")
    sample = (f"{what} (bounded sample; per-frame metric), "
              f"{args.steps} steps, {cores} of {os.cpu_count()} host threads (fastest of a probe; "
              "more threads are slower for these tensor sizes)")
    cfg, _ = workload_config(w, per_gpu, world)
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "frames_per_step_timed": frames * planes_timed / w.planes},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- #
# GPU arm                                                                     #
# --------------------------------------------------------------------------- #
def measure_gpu(w, per_gpu, steps, warmup, dev, rank, world, sampler, S, _native, sharding, variant_id):
    """value (device-resident inputs), the sweep kernel alone (roofline), and e2e (host buffers);
    `outputs`: what the last timed step returned, on the host."""
    from simplerecon_b200.pipeline import HostStreamer
    from simplerecon_b200.synthetic import make_workload_tuple, mlp_state
    hero = w.kind == "mlp"
    cfg, n_sets = workload_config(w, per_gpu, world)
    sets_host = [make_workload_tuple(w, seed_offset=1000 * rank + i, batch=per_gpu) for i in range(n_sets)]
    sets_dev = [{k: v.to(dev) for k, v in s.items()} for s in sets_host]
    with contextlib.redirect_stdout(sys.stderr):   # the managers print a banner like the reference's;
        if hero:                                   # stdout carries the ONE JSON line only
            mgr = S.FeatureVolumeManager(w.height, w.width, num_depth_bins=w.planes,
                                         mlp_channels=[0, 128, 128, 1], matching_dim_size=w.channels,
                                         num_source_views=w.views)
            mgr.load_state_dict({**mgr.state_dict(), **mlp_state(w.views, w.channels)})
        else:
            mgr = S.CostVolumeManager(w.height, w.width, num_depth_bins=w.planes)
    mgr = mgr.to(dev).eval()
    kw = dict(return_mask=True) if hero else {}
    _native.set_variant(variant_id)
    sampler.reset()
    with torch.inference_mode():
        def step(i):
            return mgr(**sets_dev[i % n_sets], **kw)

        for i in range(warmup):
            step(i)
        torch.cuda.synchronize()

        # ---- value: device-resident inputs ---------------------------------
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches0 = _native.launch_count()
        sharding.barrier()
        torch.cuda.synchronize()
        sampler.active.set()
        e0.record()
        for i in range(steps - 1):
            step(i)
        last = step(steps - 1)
        e1.record()
        torch.cuda.synchronize()
        sampler.active.clear()
        sharding.barrier()
        ms_local = e0.elapsed_time(e1)
        launches = _native.launch_count() - launches0
        ms_total = sharding.max_over_ranks(ms_local, dev)
        variant = _native.last_variant()
        clocks = sampler.snapshot()

        # ---- roofline: the sweep kernel alone, events on its own stream -----
        _native.profile_begin(steps)
        for i in range(steps):
            step(i)
        torch.cuda.synchronize()
        prep_ms, sweep_ms, nrec = _native.profile_end()

        # ---- e2e: pinned host inputs -> H2D -> sweep -> D2H, through HostStreamer ------
        pin = [{k: v.pin_memory() for k, v in s_.items()} for s_ in sets_host[:3]]
        h2d = sum(v.numel() * v.element_size() for v in pin[0].values())
        streamer = HostStreamer(mgr, dev, return_mask=hero)
        outs = list(streamer.run(pin[i % len(pin)] for i in range(6)))   # warm-up (fills the device ring)
        d2h = sum(t.numel() * t.element_size() for t in outs[-1])
        e2e_steps = max(5, min(steps, 50))
        windows = []
        for _ in range(3):
            sharding.barrier()
            torch.cuda.synchronize()
            t_wall0 = time.perf_counter()
            e0.record()
            n_out = 0
            for _host_res in streamer.run(pin[i % len(pin)] for i in range(e2e_steps)):
                n_out += 1
            e1.record()
            torch.cuda.synchronize()
            t_wall = time.perf_counter() - t_wall0
            sharding.barrier()
            assert n_out == e2e_steps
            # device time between the first H2D and the last D2H (events on the default stream bracket
            # the streamer's three streams through the synchronising yields) vs wall clock: take the
            # larger so host-side stalls are not hidden
            windows.append(sharding.max_over_ranks(max(e0.elapsed_time(e1), 1e3 * t_wall), dev))
        e2e_ms = statistics.median(windows)
    outputs = {}
    for name, t in zip(OUTPUT_NAMES, last):
        if t is None:
            continue
        if name == "depth_planes" and t.stride()[2:] == (0, 0):
            t = t[:, :, :1, :1]          # one depth per plane, broadcast over the map: (B, D, 1, 1)
        outputs[name] = t.float().cpu()
    del sets_dev, pin, streamer, mgr, last
    torch.cuda.empty_cache()

    frames_step = per_gpu * world
    sweep_s = sweep_ms * 1e-3 / max(nrec, 1)
    rec = {
        "value": frames_step * steps / (ms_total * 1e-3), "ms_per_step": ms_total / steps, "config": cfg,
        "roofline": make_roofline(w, hero, per_gpu, sweep_s, prep_ms * 1e-3 / max(nrec, 1),
                                  ms_local * 1e-3 / steps, variant, clocks.get("sm_mhz")),
        "e2e": {"value": frames_step * e2e_steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps,
                "windows_ms_per_step": [x / e2e_steps for x in windows],
                "mode": ("HostStreamer: H2D(i+1) || sweep(i) || D2H(i-1) on three streams, pinned host buffers, "
                         "persistent device input ring; median of 3 windows")},
        "gpu_launches": launches, "clocks": clocks, "kernel_variant": variant, "outputs": outputs,
    }
    return rec


def dump_outputs(directory: str, arrays: dict) -> dict:
    """Writes `arrays` as <name>.npy (float32); past DUMP_BYTES in all, each array becomes a seeded
    sample of its flattened elements, sorted by position.  Returns {name: shape, or the sample size}."""
    import numpy as np
    out = Path(directory)
    out.mkdir(parents=True, exist_ok=True)
    total = sum(4 * t.numel() for t in arrays.values())
    frac = min(1.0, DUMP_BYTES / total) if total else 1.0
    written = {}
    for name, t in arrays.items():
        a = t.numpy().astype(np.float32, copy=False)
        if frac < 1.0:
            idx = np.random.default_rng(0).choice(a.size, max(1, int(a.size * frac)), replace=False)
            a = a.reshape(-1)[np.sort(idx)]
            written[name] = f"seeded sample of {a.size} of {t.numel()} elements of {list(t.shape)}"
        else:
            written[name] = list(t.shape)
        np.save(out / f"{name}.npy", a)
    return written


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD)
    ap.add_argument("--variant", default="auto", choices=["auto", "generic", "fast"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the secondary (dot cfg1) record")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step of each workload to DIR/*.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    from simplerecon_b200.synthetic import CONFIGS, STRESS, mlp_state
    w = next(c for c in CONFIGS + STRESS if c.name.startswith(args.workload))
    per_gpu = PER_GPU.get(w.name[:4], w.batch)
    if args.impl == "reference":
        run_reference_arm(args, w, per_gpu)
        return

    import simplerecon_b200 as S
    from simplerecon_b200 import _native, sharding

    rank, world, local = sharding.init_distributed()
    if world != args.gpus and rank == 0:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE={world}", file=sys.stderr)
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (use --impl reference for the CPU arm)"
    full_affinity = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    numa_cpus = sharding.bind_to_gpu_numa(local)     # before any pinned allocation
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    _native.check(_native.load().srcv_check_device())
    variant_id = {"auto": 0, "generic": 1, "fast": 2}[args.variant]
    hero = w.kind == "mlp"

    sampler = ClockSampler(local)
    rec = measure_gpu(w, per_gpu, args.steps, args.warmup, dev, rank, world, sampler, S, _native, sharding,
                      variant_id)
    line = {
        "metric": METRIC, "value": rec["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": rec["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": rec["config"], "roofline": rec["roofline"], "e2e": rec["e2e"],
        "gpu_launches": rec["gpu_launches"], "clocks": rec["clocks"], "kernel_variant": rec["kernel_variant"],
        "host_binding": (f"{len(numa_cpus)} CPUs local to GPU {local} (NVML affinity)" if numa_cpus
                         else "none (NVML affinity unavailable)"),
    }
    if args.workload == DEFAULT_WORKLOAD and not args.no_also:
        # the dot-product configuration of BASELINE.json configs[1], same run, same clocks
        wa = next(c for c in CONFIGS if c.name.startswith(ALSO_WORKLOAD))
        ra = measure_gpu(wa, PER_GPU[ALSO_WORKLOAD], args.steps, args.warmup, dev, rank, world, sampler, S,
                         _native, sharding, variant_id)
        line["also"] = {wa.name: {k: ra[k] for k in ("value", "ms_per_step", "config", "roofline", "e2e",
                                                     "gpu_launches", "clocks", "kernel_variant")}}
    sampler.stop()
    if rank == 0 and args.dump_outputs:
        dumped = {f"{w.name.split('_')[0]}_{k}": v for k, v in rec["outputs"].items()}
        if "also" in line:
            dumped.update({f"{wa.name.split('_')[0]}_{k}": v for k, v in ra["outputs"].items()})
        line["dumped_outputs"] = {"dir": args.dump_outputs, "arrays": dump_outputs(args.dump_outputs, dumped)}

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        if full_affinity is not None:
            with contextlib.suppress(Exception):
                os.sched_setaffinity(0, full_affinity)       # the CPU leg may use every host core
        # second comparator (SURVEY.md §8d): the same port — the reference's per-plane grid_sample / cat /
        # Linear sequence — run on THIS GPU, i.e. what a user of the reference gets today on the same
        # hardware from library kernels.
        gpu_port = None
        try:
            from oracle import costvolume_oracle as O
            from simplerecon_b200.synthetic import make_workload_tuple
            frames_g = min(per_gpu, 2 if hero else 4)
            tg = {k: v.to(dev) for k, v in make_workload_tuple(w, batch=frames_g).items()}
            wg = tuple(x.to(dev) for x in O.mlp_weights_from_state_dict(mlp_state(w.views, w.channels))) if hero else None
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.inference_mode():
                cpu_port_step(w, tg, wg)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(2):
                    cpu_port_step(w, tg, wg)
                e1.record()
                torch.cuda.synchronize()
            gpu_port = {
                "value": 2 * frames_g / (e0.elapsed_time(e1) * 1e-3), "unit": UNIT,
                "sample": f"{frames_g} frame(s), 2 reps, the port's op sequence as PyTorch CUDA ops on cuda:{local}"}
        except Exception as ex:  # pragma: no cover - informational only
            gpu_port = {"value": None, "error": str(ex)[:200]}
        frames = 1 if hero else 2
        fps, cores, sample = time_cpu_port(w, frames, min_seconds=12.0, max_reps=5)
        line["cpu_baseline"] = {"value": fps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                                "port_on_this_gpu": gpu_port, "c_port_openmp": time_c_port(w, frames)}
    elif rank == 0:
        line["cpu_baseline"] = None
    if rank == 0:
        print(json.dumps(line), flush=True)
    if torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
