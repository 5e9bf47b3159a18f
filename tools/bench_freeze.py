"""Training step (config 5: Large, batch 8, 1024 x 1024, 8 classes, bf16, inputs resident in HBM, CUDA-graph replay) with
parts of the model frozen, timed alternately in one process with CUDA events:

* ``all_trainable``: the default step;
* ``all_bn_eval``: every BatchNorm in eval mode (running statistics), every parameter trainable;
* ``backbone_frozen``: the MobileNetV3 backbone's parameters ``requires_grad=False`` and its BatchNorms in eval mode;
* ``heads_only``: only ``ffm`` and ``conv_out`` train, every other parameter frozen and every other BatchNorm in eval mode.

Each setting has its own model (and its own captured graphs).  Prints ms/step, img/s and the C-ABI calls per step
(forward + backward), then one JSON line with the card's name and power limit.

    python tools/bench_freeze.py [--steps 20] [--warmup 5]
"""

import argparse
import json
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

import torch  # noqa: E402
from torch import nn  # noqa: E402

from cabinet_b200.loss import OhemCELoss  # noqa: E402
from cabinet_b200.synthetic import build_model, make_input, make_labels  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out or torch.cuda.get_device_name(0)


def freeze(model, setting):
    """Freezes parameters (requires_grad=False) and puts BatchNorms in eval mode for one setting."""
    if setting == "all_trainable":
        return
    frozen = {"all_bn_eval": (), "backbone_frozen": ("mobile",), "heads_only": ("mobile", "sb", "ab")}[setting]
    for n, m in model.named_modules():
        if isinstance(m, nn.BatchNorm2d) and (setting == "all_bn_eval" or n.startswith(frozen)):
            m.eval()
    for n, p in model.named_parameters():
        if frozen and n.startswith(frozen):
            p.requires_grad_(False)


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
    for setting in ("all_trainable", "all_bn_eval", "backbone_frozen", "heads_only"):
        m = build_model(C, "large").cuda().train()
        m.train_precision = "bf16"
        freeze(m, setting)
        models[setting] = m

    def step(m):
        m.zero_grad(set_to_none=False)
        out, out16 = m(x)
        loss = crit(out, lb) + crit(out16, lb)
        loss.backward()
        return loss.detach()

    for m in models.values():
        for _ in range(args.warmup):
            step(m)
    torch.cuda.synchronize()
    rows = []
    for rnd in range(2):
        for setting, m in models.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                loss = step(m)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / args.steps
            calls = m.train_engine().launches
            rows.append({"round": rnd, "setting": setting, "ms_per_step": round(ms, 3), "img_per_s": round(B / ms * 1e3, 1),
                         "calls_per_step": calls, "loss": round(float(loss), 5)})
            print(f"round {rnd} {setting:>15}: {ms:.3f} ms/step  {B / ms * 1e3:.1f} img/s  {calls} calls/step  "
                  f"(loss {float(loss):.5f})", flush=True)
    best = {s: min(r["ms_per_step"] for r in rows if r["setting"] == s) for s in models}
    print(json.dumps({"card": card(), "workload": f"config 5: Large, batch {B}, {H}x{W}, {C} classes, bf16, graph replay",
                      "steps": args.steps, "rows": rows, "best_ms": best}))


if __name__ == "__main__":
    main()
