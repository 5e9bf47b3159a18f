"""Time a standalone ContextAggregationBlock against eager PyTorch of the same block on the same GPU.

    python tools/bench_cab_block.py [--batch 16] [--hw 32 64] [--iters 50] [--warmup 10]

For CAB(512, 128) (the reference's unit-test width) and CAB(256, 128) (CABiNet's) at batch 16, 32 x 64 tokens: the eval
forward (``precision='bf16'``) and the train forward + backward (``train_precision='bf16'``) of the drop-in, and eager
PyTorch of the reference block (``oracle.cabinet_oracle.cab`` with fp32 weights under ``torch.autocast(bf16)``, cuDNN
benchmark on).  CUDA events around ``--iters`` calls after ``--warmup`` calls; prints the card name and power limit.
"""

from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

import torch  # noqa: E402
from torch import nn  # noqa: E402

from cabinet_b200.modules import ContextAggregationBlock  # noqa: E402
from cabinet_b200.synthetic import perturb_state_dict  # noqa: E402
from oracle import cabinet_oracle  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()),
                              "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = torch.cuda.get_device_name() + ", power limit unknown"
    return out


def timed(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def make_block(C, V):
    torch.manual_seed(0)
    blk = ContextAggregationBlock(C, V)
    for m in blk.modules():
        if isinstance(m, nn.Conv2d):
            nn.init.kaiming_normal_(m.weight, a=1)
    blk.load_state_dict(perturb_state_dict(blk.state_dict()))
    return blk.cuda()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--hw", type=int, nargs=2, default=(32, 64))
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    a = ap.parse_args()
    torch.backends.cudnn.benchmark = True
    H, W = a.hw
    rows = []
    for C, V in ((512, 128), (256, 128)):
        blk = make_block(C, V)
        x = torch.randn(a.batch, C, H, W, device="cuda")
        w = torch.randn_like(x)
        sd = {"b." + k: v for k, v in blk.state_dict().items()}
        params = {k: v.clone().requires_grad_(True) for k, v in sd.items()
                  if not k.endswith(("running_mean", "running_var", "num_batches_tracked"))}
        work = dict(sd)
        work.update(params)

        blk.eval()
        blk.precision = "bf16"
        xb = x.bfloat16()
        with torch.no_grad():
            ours_eval = timed(lambda: blk(xb), a.iters, a.warmup)

        def ref_eval():
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
                cabinet_oracle.cab(sd, "b", x)

        torch_eval = timed(ref_eval, a.iters, a.warmup)

        blk.train()
        blk.train_precision = "bf16"

        def ours_step():
            (blk(x) * w).sum().backward()

        ours_train = timed(ours_step, a.iters, a.warmup)

        def ref_step():
            cabinet_oracle.BATCH_STATS = {}
            try:
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    y = cabinet_oracle.cab(work, "b", x)
                (y.float() * w).sum().backward()
            finally:
                cabinet_oracle.BATCH_STATS = None

        torch_train = timed(ref_step, a.iters, a.warmup)
        rows.append(dict(block=f"CAB({C}, {V})", batch=a.batch, tokens=f"{H}x{W}", eval_ms=round(ours_eval, 3),
                         eval_torch_bf16_autocast_ms=round(torch_eval, 3), train_ms=round(ours_train, 3),
                         train_torch_bf16_autocast_ms=round(torch_train, 3)))
    print(json.dumps(dict(card=card(), rows=rows), indent=1))


if __name__ == "__main__":
    main()
