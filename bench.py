#!/usr/bin/env python
"""Benchmark of the CABiNet forward hot path (BASELINE.json: images/sec at 1024x1024, MNv3-Large).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|4] [--dump-outputs DIR]

``--config`` picks a BASELINE.json workload: 2 (default, the one the metric is quoted on) = Large 16x3x1024x1024, 8
classes; 3 = Large 1024x2048, 19 classes (Cityscapes shape, batch 8 per GPU); 4 = Small 2160x3840, 8 classes (UAVid 4K,
batch 4 per GPU).  ``--height/--width/--batch/--classes/--mode`` override single fields.

One process per GPU (N > 1: launched by torchrun).  A step = one forward of the hot path over one batch of
synthetic images per GPU.  Prints ONE JSON line on rank 0.

* ``value``     images/sec of ``CABiNet.forward`` (both bf16 NCHW logit tensors returned), inputs resident in HBM,
                timed with CUDA events, max over ranks.  Inputs (201 MB per batch) exceed the 126 MB L2.
* ``e2e``       the same metric through the public evaluation call with HOST buffers: pinned fp32 images ->
                H2D -> ``model.accumulate_hist`` (forward + fused upsample/argmax/confusion matrix) -> D2H of the
                uint8 mask, every step inside the timed region; the per-rank int64 confusion matrices are
                all-reduced over NCCL once at the end (the path's only collective, evaluate.py:230-235).
* ``roofline``  dominant kernel family by device time: algorithmic bytes (or flops) / CUDA-event duration of its
                launches, against MEASURED_PEAKS.json.
* ``cpu_baseline`` the oracle port of the reference forward on the host cores (rank 0, N = 1 only).
* ``gpu_eager_baseline`` the same port as eager PyTorch ON THE GPU (bf16 autocast, cudnn.benchmark, NCHW and
                channels_last, same batch): what a user of the reference gets from cuDNN/cuBLAS today (the "practical
                bar", BASELINE.md).
* ``--impl reference`` times that same CPU implementation as the reference arm.

``--dump-outputs DIR`` writes, on rank 0, what the timed path returned in its last timed step as float32
``DIR/<name>.npy``: the two logit tensors (and for ``--config 5`` the loss and the gradients).  The inputs are seeded,
so two builds run with the same arguments can be compared output for output.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "images/sec at 1024x1024 (MNv3-L)"
UNIT = "images/s"
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.is_file():
        try:
            d = json.loads(p.read_text())
            return {k: float(d[k]) for k in FALLBACK_PEAKS if k in d} | {"source": "measured"}
        except Exception:
            pass
    return dict(FALLBACK_PEAKS, source="fallback")


class ClockSampler:
    """SM clock / throttle reasons of this rank's GPU sampled WHILE the timed region runs.

    NVML polled every ~2 ms from a thread (the timed region is only tens of milliseconds long: `nvidia-smi -lms`
    cannot resolve it and its start-up alone is longer); falls back to an nvidia-smi loop if pynvml is missing."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_id: str):
        self.gpu_id, self.proc, self.lines = gpu_id, None, []
        self.samples, self.max_mhz, self.reasons, self.stop, self.nv = [], None, set(), False, None
        try:
            import pynvml

            pynvml.nvmlInit()
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(gpu_id)
            except (TypeError, AttributeError):
                self.h = pynvml.nvmlDeviceGetHandleByUUID(gpu_id.encode())
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
        except Exception:
            self.nv = None

    def _poll(self):
        nv = self.nv
        names = {getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                 getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                 getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                 getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap"}
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(
            nv, "nvmlDeviceGetCurrentClocksThrottleReasons", None)
        while not self.stop:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                if get_reasons is not None:
                    mask = int(get_reasons(self.h))
                    for bit, name in names.items():
                        if mask & bit:
                            self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def __enter__(self):
        if self.nv is not None:
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return self
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", self.gpu_id, f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.nv is not None:
            self.stop = True
            self.t.join(timeout=2)
            return
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        if self.nv is not None and self.samples:
            return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(self.reasons), "samples": len(self.samples), "source": "nvml, 2 ms period"}
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v == "Active":
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                "source": "nvidia-smi -lms 200"}


DUMP_SAMPLE = 1 << 22  # elements kept of a larger output: 16 MB in float32, so a run dumps at most 64 MB in all


def output_sample(t, n=DUMP_SAMPLE):
    """-> numpy float32 copy of ``t``: the whole tensor if it has at most ``n`` elements, else a 1-D array of the
    elements at up to ``n`` sorted flat indices drawn by a fixed seed from the element count alone, so that runs with
    the same arguments sample the same positions."""
    import numpy as np
    import torch

    t = t.detach()
    if t.numel() > n:
        idx = np.unique(np.random.default_rng(0).integers(0, t.numel(), size=n))
        t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
    return t.float().cpu().numpy()


def dump_outputs(out_dir, arrays):
    """Writes ``{name: numpy array}`` as ``out_dir/<name>.npy``."""
    import numpy as np

    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out / f"{name}.npy", a)


def cpu_forward_rate(mode, n_classes, hw, batch, iters, warmup):
    """Oracle port of the reference forward on the host cores -> (images/s, threads)."""
    import torch

    from cabinet_b200.constants import BACKBONE_CFGS
    from cabinet_b200.synthetic import build_model, make_input
    from oracle import cabinet_oracle

    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    model = build_model(n_classes, mode)
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    x = make_input(batch, hw[0], hw[1])
    times = []
    for i in range(warmup + iters):
        t0 = time.perf_counter()
        ref_out = cabinet_oracle.cabinet_forward(sd, x, BACKBONE_CFGS[mode])
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    return batch / statistics.median(times), torch.get_num_threads(), times, ref_out


def run_reference(args):
    """Reference arm: the reference's CPU implementation of the path (oracle port; the Python reference tree does
    not travel to the GPU box), all host threads, the same batch per step as our arm (``--ref-batch`` overrides)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.perf_counter()
    B = args.ref_batch or args.batch
    rate, threads, times, ref_out = cpu_forward_rate(args.mode, args.classes, (args.height, args.width), B, args.steps,
                                                     max(1, min(args.warmup, 2)))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"final_logits": output_sample(ref_out[0]), "aux_logits": output_sample(ref_out[1])})
    ms = 1e3 * statistics.median(times)
    sample = (f"{args.steps} steps x {B} images {args.height}x{args.width}, fp32, oracle port of src/models/cabinet.py "
              f"forward")
    print(json.dumps({
        "impl": "reference", "metric": metric_name(args), "value": rate, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config(args, batch=B), outputs="final + aux logits, fp32 NCHW",
                       launch="CPU: torch ops of the oracle port on all host threads",
                       cache="n/a (host)", parallelism="cpu"),
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0}))


CONFIGS = {  # BASELINE.json configs[1..4]
    2: dict(mode="large", height=1024, width=1024, batch=16, classes=8, name="BASELINE configs[1]"),
    3: dict(mode="large", height=1024, width=2048, batch=8, classes=19, name="BASELINE configs[2], Cityscapes shape"),
    4: dict(mode="small", height=2160, width=3840, batch=4, classes=8, name="BASELINE configs[3], UAVid native 4K"),
    5: dict(mode="large", height=1024, width=1024, batch=8, classes=8, name="BASELINE configs[4], training step fwd+bwd"),
}


def metric_name(args):
    if (args.height, args.width, args.mode) == (1024, 1024, "large"):
        return METRIC
    return f"images/sec at {args.height}x{args.width} (MNv3-{args.mode[0].upper()})"


def gpu_eager_rate(args, dev, iters, warmup):
    """The oracle port of the reference forward as eager PyTorch on the GPU: bf16 autocast, cudnn.benchmark, same
    batch, inputs resident -- cuDNN / cuBLAS kernels, i.e. what the reference's own ``model(x)`` costs on this B200.
    Both memory formats are timed (NCHW is what the reference runs; channels_last is the usual eager tuning)."""
    import torch

    from cabinet_b200.constants import BACKBONE_CFGS
    from cabinet_b200.synthetic import build_model, make_input
    from oracle import cabinet_oracle

    model = build_model(args.classes, args.mode)
    x0 = make_input(args.batch, args.height, args.width).to(dev)
    prev = torch.backends.cudnn.benchmark
    torch.backends.cudnn.benchmark = True
    out = {"unit": UNIT, "batch": args.batch, "dtype": "bf16 autocast", "impl": "eager PyTorch (cuDNN/cuBLAS), oracle port "
           "of src/models/cabinet.py:207-247", "variants": {}}
    try:
        for fmt in ("nchw", "channels_last"):
            try:
                cl = fmt == "channels_last"
                sd = {k: v.to(dev) for k, v in model.state_dict().items()}
                if cl:
                    sd = {k: (v.contiguous(memory_format=torch.channels_last) if v.dim() == 4 else v) for k, v in sd.items()}
                x = x0.contiguous(memory_format=torch.channels_last) if cl else x0
                with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
                    for _ in range(warmup):
                        cabinet_oracle.cabinet_forward_graph(sd, x, BACKBONE_CFGS[args.mode])
                    torch.cuda.synchronize(dev)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(iters):
                        cabinet_oracle.cabinet_forward_graph(sd, x, BACKBONE_CFGS[args.mode])
                    e1.record()
                    torch.cuda.synchronize(dev)
                ms = e0.elapsed_time(e1) / iters
                out["variants"][fmt] = {"value": args.batch / (ms * 1e-3), "ms_per_step": ms}
            except Exception as err:  # e.g. a .view() of the reference's attention code on a channels_last tensor
                out["variants"][fmt] = {"error": f"{type(err).__name__}: {str(err)[:160]}"}
            torch.cuda.empty_cache()
    finally:
        torch.backends.cudnn.benchmark = prev
    ok = {k: v for k, v in out["variants"].items() if "value" in v}
    if ok:
        best = max(ok, key=lambda k: ok[k]["value"])
        out.update(value=ok[best]["value"], ms_per_step=ok[best]["ms_per_step"], memory_format=best)
    return out


def h2d_ceiling_gbs(dev, nbytes=256 << 20, iters=6):
    """Measured pinned host -> device copy rate of this rank (all ranks run it at the same time, so at N > 1 it is
    the per-GPU share of the host's aggregate rate): the ceiling of any end-to-end number fed from host memory."""
    import torch

    src = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    dst = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        dst.copy_(src, non_blocking=True)
    e1.record()
    torch.cuda.synchronize(dev)
    return nbytes * iters / (e0.elapsed_time(e1) * 1e-3) / 1e9


def workload_config(args, batch=None):
    B = batch or args.batch
    in_mb = B * 3 * args.height * args.width * 4 / 1e6
    return {"workload": f"CABiNet MobileNetV3-{args.mode.capitalize()} forward, {args.height}x{args.width}, "
                        f"batch {B} per GPU, {args.classes} classes ({args.config_name})",
            "mode": args.mode, "size": args.height if args.height == args.width else [args.height, args.width],
            "batch_per_gpu": B, "n_classes": args.classes,
            "outputs": "final + aux logits, bf16 NCHW", "launch": "CUDA graph replay of the kernel schedule",
            "cache": f"inputs ({in_mb:.0f} MB/batch) larger than the 126 MB L2" if in_mb > 126 else
                     f"inputs {in_mb:.0f} MB/batch; every layer's activations ({B} images) exceed the 126 MB L2 several times over",
            "weights": "random-init seed 0 + perturbed BN/bias/gamma (synthetic.py)", "parallelism": f"dp{args.gpus}"}


def summarise_trace(rows, steps, peaks):
    """Per-kernel-family totals -> table + the dominant family's roofline entry."""
    fam = {}
    for r in rows:
        f = fam.setdefault(r["kernel"], {"ms": 0.0, "bytes": 0, "fused_bytes": 0, "flops": 0, "launches": 0})
        f["ms"] += r["ms"]
        f["bytes"] += r["bytes"]
        f["fused_bytes"] += r.get("fused_bytes", r["bytes"])
        f["flops"] += r["flops"]
        f["launches"] += 1
    total = sum(f["ms"] for f in fam.values()) or 1.0
    table = []
    for k, f in sorted(fam.items(), key=lambda kv: -kv[1]["ms"]):
        gbs = f["bytes"] / (f["ms"] * 1e-3) / 1e9 if f["ms"] else 0.0
        tfl = f["flops"] / (f["ms"] * 1e-3) / 1e12 if f["ms"] else 0.0
        row = {"kernel": k, "share": f["ms"] / total, "ms_per_step": f["ms"] / steps,
               "launches_per_step": f["launches"] / steps, "GB/s": gbs, "TFLOP/s": tfl}
        if f["fused_bytes"] != f["bytes"]:
            # block-fused kernels: "GB/s" counts SURVEY 8(d)'s per-layer-fusion bytes (the expanded tensors they keep on
            # chip included); this is the traffic the kernel itself has to move
            row["block_fused_GB/s"] = f["fused_bytes"] / (f["ms"] * 1e-3) / 1e9 if f["ms"] else 0.0
        table.append(row)
    return table


def roofline_by_bound(fam_rows, peaks):
    """The dominant family mixes HBM-bound and tensor-bound layers (conv_tc runs the 1x1 convs and the dense 3x3
    convs): classify every launch by its own floor max(bytes / HBM peak, flops / tensor peak) and report each class
    against its own peak, plus the share of the family's time that the per-launch floors explain."""
    tf_peak, hbm = peaks["bf16_tflops_sustained"], peaks["hbm_gbs"]
    cls = {"hbm": {"ms": 0.0, "bytes": 0, "flops": 0, "launches": 0, "floor_ms": 0.0},
           "tensor": {"ms": 0.0, "bytes": 0, "flops": 0, "launches": 0, "floor_ms": 0.0}}
    for r in fam_rows:
        t_hbm, t_tc = r["bytes"] / (hbm * 1e9), r["flops"] / (tf_peak * 1e12)
        c = cls["tensor" if t_tc > t_hbm else "hbm"]
        c["ms"] += r["ms"]
        c["bytes"] += r["bytes"]
        c["flops"] += r["flops"]
        c["launches"] += 1
        c["floor_ms"] += 1e3 * max(t_hbm, t_tc)
    out = {}
    for name, c in cls.items():
        if not c["launches"]:
            continue
        if name == "hbm":
            ach, peak, unit = c["bytes"] / (c["ms"] * 1e-3) / 1e9, hbm, "GB/s"
        else:
            ach, peak, unit = c["flops"] / (c["ms"] * 1e-3) / 1e12, tf_peak, "TFLOP/s"
        out[name] = {"achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak, "launches": c["launches"],
                     "time_share_of_family": c["ms"] / sum(v["ms"] for v in cls.values())}
    total = sum(v["ms"] for v in cls.values())
    out["floor_frac"] = sum(v["floor_ms"] for v in cls.values()) / total if total else None
    return out


def ncu_traffic_per_launch(kernel, args, positions=None):
    """dram read+write bytes per launch of a kernel family from the committed ncu capture of this workload
    (profiles/r02_ncu_dram_traffic_per_family.json: one forward, batch 16, Large, 1024x1024), else None.
    ``positions``: indices (schedule order inside one forward) of the family's launches to average over."""
    p = ROOT / "profiles" / "r02_ncu_dram_traffic_per_family.json"
    if not p.is_file() or (args.batch, args.height, args.width, args.mode, args.classes) != (16, 1024, 1024, "large", 8):
        return None
    try:
        fam = json.loads(p.read_text())["families"]
        for name, f in fam.items():
            if name.startswith(kernel):
                per = f.get("per_launch_dram_bytes")
                if positions and per and max(positions) < len(per):
                    return sum(per[i] for i in positions) / len(positions)
                return (f["dram_read_bytes"] + f["dram_write_bytes"]) / f["launches"]
    except Exception:
        pass
    return None


def roofline_entry(row, fam_rows, peaks, timed_in_step=True):
    nbytes = sum(r["bytes"] for r in fam_rows)
    flops = sum(r["flops"] for r in fam_rows)
    ms = sum(r["ms"] for r in fam_rows)
    n = len(fam_rows)
    tf_peak = peaks["bf16_tflops_sustained" if timed_in_step else "bf16_tflops"]
    t_hbm = nbytes / (peaks["hbm_gbs"] * 1e9)
    t_tc = flops / (tf_peak * 1e12)
    if t_tc > t_hbm:
        ach = flops / (ms * 1e-3) / 1e12
        return {"kernel": row["kernel"], "bound": "tensor", "achieved": ach, "peak": tf_peak, "unit": "TFLOP/s",
                "frac": ach / tf_peak, "traffic": None, "launches": n, "avg_launch_us": 1e3 * ms / n,
                "algorithmic_flops_per_launch": flops / n, "peak_source": peaks["source"]}
    ach = nbytes / (ms * 1e-3) / 1e9
    return {"kernel": row["kernel"], "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": ach / peaks["hbm_gbs"], "traffic": None, "launches": n, "avg_launch_us": 1e3 * ms / n,
            "algorithmic_bytes_per_launch": nbytes / n, "peak_source": peaks["source"]}


def run_ours(args):
    import torch
    import torch.distributed as dist

    from cabinet_b200.synthetic import build_model, make_input, make_labels

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = {"bound": False, "why": "--no-numa-bind" if args.no_numa_bind else "single rank: all host cores stay available "
            "to the cpu_baseline leg"}
    if not args.no_numa_bind and world > 1:
        # before any pinned allocation: the rank's host buffers are first-touched on its GPU's NUMA node
        from cabinet_b200.affinity import bind_to_gpu_numa

        numa = bind_to_gpu_numa(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()
    K, Wm, B, C = args.steps, args.warmup, args.batch, args.classes
    H, W = args.height, args.width

    model = build_model(C, args.mode).to(dev)
    model.precision = args.precision
    model.logits_dtype = torch.bfloat16
    model.use_cuda_graph = not args.no_graph  # replay the captured kernel schedule (immune to host launch jitter)
    eng = model.engine()
    x_host = make_input(B, H, W, seed=7 + rank).pin_memory()          # each rank owns different images
    lb_host = make_labels(B, H, W, C, seed=11 + rank).to(torch.uint8).pin_memory()
    x = x_host.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    uuid = str(torch.cuda.get_device_properties(local).uuid)
    gpu_id = uuid if uuid.startswith("GPU-") else "GPU-" + uuid

    # ---------------- device-resident throughput (value)
    with torch.no_grad():
        # W warm-up steps + 2 priming replays: the engine captures the graph on the caller's buffer at its third
        # sighting, and the first replay of a fresh graph pays its upload
        for _ in range(Wm + 2):
            model(x)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(gpu_id) as clk:
            e0.record()
            for _ in range(K):
                out = model(x)
            e1.record()
            barrier()
        launches = eng.launches * K
        ms_total = max_over_ranks(e0.elapsed_time(e1))
        value = world * B * K / (ms_total * 1e-3)
        clocks = clk.summary()
        gpu_img0 = (out[0][:1].float().cpu(), out[1][:1].float().cpu())  # image 0: compared with the oracle below
        # the graph's static output buffers: sampled now, before the traced steps below overwrite them
        dumped = None
        if args.dump_outputs and rank == 0:
            dumped = {"final_logits": output_sample(out[0]), "aux_logits": output_sample(out[1])}
        del out

        # ---------------- per-kernel roofline: same K steps, every launch bracketed by CUDA events on its stream
        eng.start_trace()
        for _ in range(K):
            model(x)
        rows = eng.stop_trace()
        table = summarise_trace(rows, K, peaks)
        dom = table[0]
        roof = roofline_entry(dom, [r for r in rows if r["kernel"] == dom["kernel"]], peaks)
        fam_rows = [r for r in rows if r["kernel"] == dom["kernel"]]
        roof["by_bound"] = roofline_by_bound(fam_rows, peaks)
        # The family mixes HBM-bound and tensor-bound layers: the headline entry is the class that holds most of the
        # family's device time (each launch classified by its own floor); the whole-family aggregate stays alongside.
        cls = max(("hbm", "tensor"), key=lambda c: roof["by_bound"].get(c, {}).get("time_share_of_family", 0.0))
        c = roof["by_bound"][cls]
        crow = [r for r in fam_rows if (r["flops"] / (peaks["bf16_tflops_sustained"] * 1e12) > r["bytes"] / (peaks["hbm_gbs"] * 1e9)) == (cls == "tensor")]
        roof["family_aggregate"] = {k: roof[k] for k in ("bound", "achieved", "peak", "unit", "frac", "launches", "avg_launch_us")}
        roof.update(bound=cls, achieved=c["achieved"], peak=c["peak"], unit=c["unit"], frac=c["frac"], launches=len(crow),
                    avg_launch_us=1e3 * sum(r["ms"] for r in crow) / len(crow),
                    launch_class=f"{dom['kernel']} launches whose own floor is {cls}-bound "
                                 f"({c['time_share_of_family']:.0%} of the family's device time)")
        roof.pop("algorithmic_flops_per_launch", None)
        roof.pop("algorithmic_bytes_per_launch", None)
        roof["algorithmic_" + ("bytes" if cls == "hbm" else "flops") + "_per_launch"] = (
            sum(r["bytes" if cls == "hbm" else "flops"] for r in crow) / len(crow))
        per_step = len(fam_rows) // K
        cls_pos = [i for i, r in enumerate(fam_rows[:per_step]) if r in crow]
        if any(r.get("fused_bytes", r["bytes"]) != r["bytes"] for r in crow):
            roof["block_fused_bytes_per_launch"] = sum(r.get("fused_bytes", r["bytes"]) for r in crow) / len(crow)
            roof["bytes_definition"] = ("algorithmic bytes = SURVEY 8(d) per-layer-fusion model (each conv of the block reads "
                                        "its input / writes its output once); block_fused_bytes_per_launch = what the fused "
                                        "kernel has to move (the expanded tensors stay on chip)")
        roof["traffic"] = ncu_traffic_per_launch(dom["kernel"], args, cls_pos)
        roof["traffic_source"] = "profiles/r02_ncu_dram_traffic_per_family.json (ncu dram__bytes_read+write per launch)"
        traced_ms = sum(r["ms"] for r in rows) / K

        # ---------------- end to end through the public evaluation call, host buffers
        # cabinet_b200.evaluator.MscEvalV0 (mirror of the reference evaluator, evaluate.py:193-253) over K pinned host
        # batches: per step H2D of the images + uint8 labels, fused forward/upsample/argmax/confusion matrix, D2H of the
        # step's result (the running int64 confusion matrix); copies run ahead of the forward on a second stream; the
        # per-rank matrices are all-reduced over NCCL at the end and the metrics are read back (inside the timed region).
        # Three feeds: fp32 NCHW host tensors (the reference loader's contract: the headline `e2e`), raw uint8 NHWC
        # images normalised on the device (SURVEY 8f-2: 3 instead of 12 bytes per pixel cross PCIe), and the fp32 feed
        # with the uint8 mask of every batch read back as well (what round 1 reported).
        from cabinet_b200.evaluator import MscEvalV0

        crop = H if H == W else (H, W)
        u8_host = torch.randint(0, 256, (B, H, W, 3), dtype=torch.uint8,
                                generator=torch.Generator().manual_seed(21 + rank)).pin_memory()
        trace = torch.zeros((K, C, C), dtype=torch.int64).pin_memory()
        masks = [torch.empty((B, H, W), dtype=torch.uint8).pin_memory() for _ in range(K)]  # D2H targets, allocated up front
        valid = int((lb_host != 255).sum()) * K
        h2d_gbs = h2d_ceiling_gbs(dev)

        def run_e2e(images, with_masks):
            ev = MscEvalV0(model, [(images, lb_host)] * 4, C, 255, (1.0,), False, cropsize=crop)
            kw = dict(masks_out=masks) if with_masks else dict(hist_trace=trace)
            for _ in range(2):  # warm-up (8 batches): ring buffers, captured graphs of the fused call, first replays
                ev.evaluate(**kw)
            ev.dl = [(images, lb_host)] * K
            barrier()
            t0 = time.perf_counter()
            e0.record()
            res = ev.evaluate(**kw)
            e1.record()
            barrier()
            wall = time.perf_counter() - t0
            ms = max_over_ranks(max(e0.elapsed_time(e1), 0.0))
            h2d = images.numel() * images.element_size() + lb_host.numel()
            return {"value": world * B * K / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": masks[0].numel() if with_masks else 8 * C * C, "ms_per_step": ms / K,
                    "wall_s": wall, "h2d_gbs_achieved": h2d * K / (ms * 1e-3) / 1e9,
                    "hist_checksum_ok": (world > 1) or int(res["confusion_matrix"].sum()) == valid}, res

        e2e, res = run_e2e(x_host, False)
        # the running matrix read back after the last step equals this rank's final matrix (before the all-reduce)
        e2e["step_result_readback_ok"] = bool(world > 1 or int(trace[K - 1].sum()) == valid)
        e2e8, _ = run_e2e(u8_host, False)
        e2e_masks, _ = run_e2e(x_host, True)
        # parity of the end-to-end result on a small sample: the confusion matrix of the evaluator call == the oracle's
        # compute_hist (numpy bincount, evaluate.py:162-191) of the masks it read back
        from oracle.evaluator_oracle import compute_hist
        nchk = min(2, B)
        hist_dev = torch.zeros((C, C), dtype=torch.int64, device=dev)
        m_dev = model.accumulate_hist(x[:nchk].contiguous(), lb_host[:nchk].to(dev), hist_dev)
        want = sum(compute_hist(m_dev[i].cpu().numpy(), lb_host[i].numpy(), C, 255) for i in range(nchk))
        e2e["hist_equals_oracle_compute_hist"] = bool((hist_dev.cpu().numpy() == want).all())
        e2e.update(
            api="cabinet_b200.evaluator.MscEvalV0.evaluate: pinned fp32 NCHW host batches, H2D ahead of the fused "
                "forward + upsample/argmax/confusion matrix, per-step D2H of the running matrix, NCCL all-reduce, metrics",
            mIoU=float(res["mIoU"]), h2d_ceiling_gbs_measured=h2d_gbs,
            h2d_bound_value=world * B / ((x_host.numel() * 4 + lb_host.numel()) / (h2d_gbs * 1e9)),
            uint8_value=e2e8["value"], uint8_ms_per_step=e2e8["ms_per_step"], uint8_h2d_bytes_per_step=e2e8["h2d_bytes_per_step"],
            uint8_frac_of_device_value=e2e8["value"] / value, with_mask_readback_value=e2e_masks["value"],
            note="fp32 host input is PCIe-bound (h2d_bound_value); uint8_value = same call fed uint8 NHWC images")
        e2e8["input"] = "uint8 NHWC images + uint8 labels, normalised on the device (cabinet_normalize_u8)"

        # ---------------- the reference's default evaluation protocol (configs/train.yaml:65-66: six scales + flip TTA,
        # sliding 1024^2 windows, stride 853): 30 class-map forwards per batch + the fused softmax / window / resize /
        # argmax / confusion-matrix kernels, next to the same evaluator taking the reference's steps as torch ops.
        msflip = None
        if args.msflip and world == 1 and H == W:
            bm = min(B, args.msflip)
            scales = (0.5, 0.75, 1.0, 1.25, 1.5, 1.75)
            evm = MscEvalV0(model, [(x_host[:bm], lb_host[:bm])], C, 255, scales, True, cropsize=H)
            msflip = {"unit": UNIT, "batch": bm, "scales": list(scales), "flip": True,
                      "forwards_per_batch": 30, "h2d_bytes_per_step": bm * (3 * H * W * 4 + H * W)}
            hists = {}
            for name, fused in (("fused_kernels", True), ("torch_ops", False)):
                evm.fused_general = fused
                for _ in range(2):
                    evm.evaluate()
                barrier()
                e0.record()
                r = evm.evaluate()
                e1.record()
                barrier()
                hists[name] = r["confusion_matrix"]
                msflip[name] = {"value": bm / (e0.elapsed_time(e1) * 1e-3), "ms_per_batch": e0.elapsed_time(e1)}
            msflip["value"] = msflip["fused_kernels"]["value"]
            msflip["pixels_differing_between_paths"] = float(abs(hists["fused_kernels"] - hists["torch_ops"]).sum() / 2
                                                             / max(hists["torch_ops"].sum(), 1))
            del evm
            torch.cuda.empty_cache()

        # ---------------- the practical bar: the reference forward as eager PyTorch on this GPU
        eager = None
        if world == 1 and not args.no_gpu_eager:
            torch.cuda.empty_cache()
            eager = gpu_eager_rate(args, dev, max(3, min(K, 10)), 3)

    if world > 1:
        dist.destroy_process_group()
    if rank != 0:
        return
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)

    # whole-forward roofline: SURVEY 8(d)'s per-layer-fusion algorithmic bytes per image (two bf16 logit tensors returned)
    # x the batch / the step time; the engine's own per-launch byte count (block-fused kernels move less) alongside
    survey_mb = {("large", 1024, 1024): 610.9, ("large", 1024, 2048): 1300.3, ("small", 2160, 3840): 2619.2}
    fused_bytes = sum(r.get("fused_bytes", r["bytes"]) for r in rows) / K
    step_bytes = survey_mb.get((args.mode, H, W), 0.0) * 1e6 * B or fused_bytes
    step_flops = sum(r["flops"] for r in rows) / K
    bb = roof["by_bound"]
    roof.update(
        hbm_class_frac=bb.get("hbm", {}).get("frac"), hbm_class_gbs=bb.get("hbm", {}).get("achieved"),
        tensor_class_frac=bb.get("tensor", {}).get("frac"), tensor_class_tflops=bb.get("tensor", {}).get("achieved"),
        floor_frac_of_family_time=bb.get("floor_frac"),
        whole_forward_gbs=step_bytes / (ms_total / K * 1e-3) / 1e9,
        whole_forward_frac=step_bytes / (ms_total / K * 1e-3) / 1e9 / peaks["hbm_gbs"],
        whole_forward_algorithmic_bytes=step_bytes, whole_forward_block_fused_bytes=fused_bytes,
        whole_forward_flops=step_flops)
    line = {
        "metric": metric_name(args), "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
        "config": workload_config(args),
        "e2e": e2e, "e2e_uint8": e2e8, "e2e_with_mask_readback": e2e_masks, "e2e_multiscale_flip": msflip,
        "gpu_launches": launches, "clocks": clocks, "numa": numa, "roofline": roof,
        "kernels": table, "traced_ms_per_step": traced_ms, "peaks": peaks,
    }
    if eager is not None:
        line["gpu_eager_baseline"] = eager
    if world == 1 and not args.no_cpu_baseline:
        rate, threads, times, ref_out = cpu_forward_rate(args.mode, C, (H, W), 1, args.cpu_iters, 3)
        # parity of this very run: image 0 of the timed batch (the oracle's input is the same first image) against the
        # oracle's fp32 forward -- the north star's bars are 1e-2 relative on the logits, masks >= 99.9 % on pixels whose
        # fp32 margin exceeds the bf16 error bar (raw agreement reported too)
        f_ref, a_ref = ref_out[0].float(), ref_out[1].float()
        f, a = gpu_img0
        top2 = f_ref.topk(2, dim=1).values
        sure = (top2[:, 0] - top2[:, 1]) > 4e-2 * float(f_ref.abs().max())
        same = f.argmax(1) == f_ref.argmax(1)
        line["parity_sample"] = {
            "image": "image 0 of the timed batch vs the oracle port (fp32, CPU) on the same weights and input",
            "final_rel_l2": float((f - f_ref).norm() / f_ref.norm()), "aux_rel_l2": float((a - a_ref).norm() / a_ref.norm()),
            "mask_agreement_raw": float(same.float().mean()),
            "mask_agreement_margin_filtered": float(same[sure].float().mean()) if bool(sure.any()) else None,
            "margin_filtered_pixel_share": float(sure.float().mean())}
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": f"{len(times)} timed forwards of 1 image {H}x{W} fp32 (median), oracle port of "
                                          f"the reference forward, {sum(times):.1f} s of CPU work on {threads} threads"}
        if eager is not None and "value" in eager:  # scalars inside a key the driver parses
            line["cpu_baseline"].update(gpu_eager_value=eager["value"], gpu_eager_ms_per_step=eager["ms_per_step"],
                                        gpu_eager_memory_format=eager["memory_format"],
                                        value_over_gpu_eager=value / eager["value"])
    print(json.dumps(line))


def run_train(args):
    """BASELINE configs[4]: Large training step (train-mode forward, 2 x OhemCELoss, backward, bucketed gradient
    all-reduce over NCCL), batch 8 per GPU.  ``value`` = images/s with inputs resident in HBM; ``e2e`` = the same step
    fed from pinned host memory (H2D of images + labels, D2H of the loss) every step."""
    import torch
    import torch.distributed as dist

    from cabinet_b200.grad_sync import GradBuckets
    from cabinet_b200.loss import OhemCELoss
    from cabinet_b200.synthetic import build_model, make_input, make_labels

    rank, world, local = (int(os.environ.get(k, d)) for k, d in (("RANK", "0"), ("WORLD_SIZE", "1"), ("LOCAL_RANK", "0")))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    K, Wm, B, C, H, W = args.steps, args.warmup, args.batch, args.classes, args.height, args.width
    model = build_model(C, args.mode).to(dev).train()
    model.train_precision = args.train_precision
    model.logits_dtype = torch.bfloat16 if args.train_precision == "bf16" else torch.float32
    crit_p, crit_16 = OhemCELoss(0.7, B * H * W // 16, 255), OhemCELoss(0.7, B * H * W // 16, 255)  # configs/train.yaml
    gb = GradBuckets(model.named_parameters())
    x_host = make_input(B, H, W, seed=7 + rank).pin_memory()
    lb_host = make_labels(B, H, W, C, seed=11 + rank).pin_memory()
    x, lb = x_host.to(dev), lb_host.to(dev)
    eng = model.train_engine()
    last = {}  # logits of the last timed step (--dump-outputs)

    def step(xd, ld, keep=False):
        gb.zero_()
        out, out16 = model(xd)
        if keep:
            last.update(final_logits=out, aux_logits=out16)
        loss = crit_p(out, ld) + crit_16(out16, ld)
        loss.backward()
        if not os.environ.get("CABINET_BENCH_NO_GRAD_SYNC"):  # diagnostic: independent replicas (max over ranks without NCCL)
            gb.all_reduce()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    uuid = str(torch.cuda.get_device_properties(local).uuid)
    gpu_id = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
    for _ in range(Wm):
        step(x, lb)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    with ClockSampler(gpu_id) as clk:
        e0.record()
        for i in range(K):
            loss = step(x, lb, keep=bool(args.dump_outputs) and i == K - 1)
            launches += eng.launches
        e1.record()
        barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    value = world * B * K / (ms * 1e-3)
    dumped = None
    if args.dump_outputs and rank == 0:  # before the steps below overwrite the gradients
        grads = torch.cat([p.grad.reshape(-1) for p in model.parameters() if p.grad is not None])
        dumped = {"loss": output_sample(loss), **{k: output_sample(v) for k, v in last.items()},
                  "gradients": output_sample(grads)}
        del grads
    # end to end: host batch in, loss out, every step
    from cabinet_b200.prefetch import DevicePrefetcher

    feed = DevicePrefetcher([(x_host, lb_host)] * K, dev)  # copies of batch i + 1 run under step i
    for i, (xd, ld) in enumerate(feed):  # untimed: the side stream's allocator pool
        step(xd, ld)
        if i == 1:
            break
    barrier()
    e0.record()
    for xd, ld in feed:
        lv = float(step(xd, ld).item())
    e1.record()
    barrier()
    e2e_ms = max_over_ranks(e0.elapsed_time(e1))
    # per-kernel shares of one traced step
    eng.start_trace()
    step(x, lb)
    rows = eng.stop_trace()
    fam = {}
    for n, ph, t in rows:
        f = fam.setdefault((n.replace("cabinet_", ""), ph), [0.0, 0])
        f[0] += t
        f[1] += 1
    table = [{"kernel": k, "phase": ph, "ms_per_step": v[0], "launches_per_step": v[1]}
             for (k, ph), v in sorted(fam.items(), key=lambda kv: -kv[1][0])]
    # roofline of the dominant kernel: the convolution gradients (and the forward convolutions of this mode) are
    # implicit GEMMs; their algorithmic FLOPs are ~3x the forward's (SURVEY 8d config 5)
    peaks = load_peaks()
    fwd_flops = 54.31e9 * B if (args.mode, H, W) == ("large", 1024, 1024) else None
    dom = table[0]
    conv_ms = sum(r["ms_per_step"] for r in table if r["kernel"] in ("conv_wgrad", "conv_dgrad", "conv2d_simt", "conv_tc"))
    roof = {"kernel": dom["kernel"], "bound": "tensor", "unit": "TFLOP/s", "peak": peaks["bf16_tflops_sustained"],
            "peak_source": peaks["source"], "traffic": None,
            "achieved": (3 * fwd_flops / (conv_ms * 1e-3) / 1e12) if fwd_flops and conv_ms else None,
            "note": "dense convolution forward + data + weight gradients (3 x 54.31 GFLOP / image) over their summed device time; "
                    "fp32 mode runs them as CUDA-core implicit GEMMs"}
    roof["frac"] = roof["achieved"] / roof["peak"] if roof["achieved"] else None
    # the practical bar: the same step as eager PyTorch on this GPU (oracle restatement of the reference: functional
    # forward with train-mode F.batch_norm, sort-based OHEM, autograd), bf16 autocast + cudnn.benchmark
    eager = None
    if world == 1 and not args.no_gpu_eager:
        del loss
        gb.zero_()
        torch.cuda.empty_cache()
        try:
            from cabinet_b200.constants import BACKBONE_CFGS
            from oracle.train_oracle import train_step as oracle_step

            sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
            prev = torch.backends.cudnn.benchmark
            torch.backends.cudnn.benchmark = True
            n_min = B * H * W // 16
            with torch.autocast("cuda", dtype=torch.bfloat16):
                for _ in range(3):
                    oracle_step(sd, x, lb, BACKBONE_CFGS[args.mode], 0.7, n_min)
                torch.cuda.synchronize(dev)
                e0.record()
                for _ in range(max(3, min(K, 5))):
                    oracle_step(sd, x, lb, BACKBONE_CFGS[args.mode], 0.7, n_min)
                e1.record()
                torch.cuda.synchronize(dev)
            torch.backends.cudnn.benchmark = prev
            ems = e0.elapsed_time(e1) / max(3, min(K, 5))
            eager = {"value": B / (ems * 1e-3), "unit": UNIT, "ms_per_step": ems, "dtype": "bf16 autocast",
                     "impl": "eager PyTorch autograd (cuDNN/cuBLAS) of the oracle train step, NCHW"}
        except Exception as err:
            eager = {"error": f"{type(err).__name__}: {str(err)[:200]}"}
    if world > 1:
        dist.destroy_process_group()
    if rank != 0:
        return
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    n_grad = sum(b.numel() for b in gb.buckets)
    print(json.dumps({
        "metric": "training images/sec at 1024x1024 (MNv3-L), fwd+bwd" if (H, W, args.mode) == (1024, 1024, "large")
        else f"training images/sec at {H}x{W} (MNv3-{args.mode[0].upper()}), fwd+bwd",
        "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": ms / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if args.train_precision == "bf16" else "f32", "data": "synthetic",
        "config": dict(workload_config(args), outputs="loss + gradients of 398 parameter tensors",
                       launch="two CUDA graphs (forward, backward) of C-ABI kernel launches, replayed per step after 2 eager steps",
                       cache="activations of a step far exceed the 126 MB L2",
                       loss="2 x OhemCELoss(thresh 0.7, n_min = pixels / 16)", grad_elements=n_grad,
                       grad_sync=f"{len(gb.buckets)} flat fp32 buckets, one async NCCL all-reduce each"),
        "e2e": {"value": world * B * K / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms / K,
                "h2d_bytes_per_step": x_host.numel() * 4 + lb_host.numel() * 8, "d2h_bytes_per_step": 4,
                "api": "DevicePrefetcher(pinned host batches) -> model.train()(x) -> OhemCELoss x 2 -> loss.backward() -> GradBuckets.all_reduce()", "loss": lv},
        "gpu_launches": launches, "clocks": clk.summary(), "roofline": roof, "kernels": table[:14],
        "traced_ms_per_step": sum(t for _, _, t in rows), "gpu_eager_baseline": eager}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="BASELINE.json workload (2 = headline)")
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--size", type=int, default=None, help="square input (sets --height and --width)")
    ap.add_argument("--height", type=int, default=None)
    ap.add_argument("--width", type=int, default=None)
    ap.add_argument("--mode", default=None, choices=["large", "small"])
    ap.add_argument("--classes", type=int, default=None)
    ap.add_argument("--ref-batch", type=int, default=0, help="--impl reference: images per step (default: --batch)")
    ap.add_argument("--cpu-iters", type=int, default=None, help="timed forwards of the cpu_baseline leg")
    ap.add_argument("--no-gpu-eager", action="store_true")
    ap.add_argument("--train-precision", default="fp32", choices=["fp32", "bf16"], help="--config 5: activation dtype")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--msflip", type=int, default=4, help="batch of the multi-scale + flip evaluation leg (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (at most 64 MB, seeded sample)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    cfg = CONFIGS[args.config]
    if args.size:
        args.height = args.height or args.size
        args.width = args.width or args.size
    for k in ("mode", "height", "width", "batch", "classes"):
        if getattr(args, k) is None:
            setattr(args, k, cfg[k])
    custom = any(getattr(args, k) != cfg[k] for k in ("mode", "height", "width", "batch", "classes"))
    args.config_name = cfg["name"] + (" (modified)" if custom else "")
    if args.cpu_iters is None:  # ~10-30 s of CPU work whatever the image size
        args.cpu_iters = max(5, min(60, int(60 * 1024 * 1024 / (args.height * args.width))))
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    elif args.config == 5:
        run_train(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
