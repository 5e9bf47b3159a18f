"""Training step (config 5: Large, batch 8, 1024 x 1024, 8 classes, inputs resident in HBM, CUDA-graph replay) in the bf16
and the fp16 training modes, timed alternately in one process (bf16, fp16, bf16, fp16) with CUDA events.

Both modes return fp32 logits (the default ``logits_dtype``), so the two rows differ in the activation type only.

    python tools/bench_train_precision.py [--steps 20] [--warmup 5]
"""

import argparse
import json
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

import torch  # noqa: E402

from cabinet_b200.loss import OhemCELoss  # noqa: E402
from cabinet_b200.synthetic import build_model, make_input, make_labels  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out or torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--size", type=int, default=1024)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    assert args.steps >= 10 and args.warmup >= 3, "time >= 10 steps after >= 3 warm-up steps (graph capture at step 3)"
    B, H, W, C = args.batch, args.size, args.size, 8
    x, lb = make_input(B, H, W, seed=7).cuda(), make_labels(B, H, W, C, seed=11).cuda()
    crit = OhemCELoss(0.7, B * H * W // 16, 255)
    models = {}
    for precision in ("bf16", "fp16"):
        m = build_model(C, "large").cuda().train()
        m.train_precision = precision
        models[precision] = m

    def step(m):
        m.zero_grad(set_to_none=False)
        out, out16 = m(x)
        loss = crit(out, lb) + crit(out16, lb)
        loss.backward()
        return loss

    for m in models.values():
        for _ in range(args.warmup):
            step(m)
    torch.cuda.synchronize()
    rows = []
    for rnd in range(2):
        for precision, m in models.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                loss = step(m)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / args.steps
            rows.append({"round": rnd, "precision": precision, "ms_per_step": round(ms, 3), "img_per_s": round(B / ms * 1e3, 1),
                         "loss": round(float(loss), 5)})
            print(f"round {rnd} {precision}: {ms:.3f} ms/step  {B / ms * 1e3:.1f} img/s  (loss {float(loss):.5f})", flush=True)
    best = {p: min(r["ms_per_step"] for r in rows if r["precision"] == p) for p in models}
    print(json.dumps({"card": card(), "workload": f"config 5: Large, batch {B}, {H}x{W}, {C} classes, graph replay",
                      "steps": args.steps, "rows": rows, "best_ms": best,
                      "fp16_vs_bf16": round(best["fp16"] / best["bf16"] - 1.0, 4)}))


if __name__ == "__main__":
    main()
