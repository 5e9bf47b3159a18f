"""Input gradients at config-5 geometry (Large, batch 8, 1024 x 1024, 8 classes, bf16, inputs resident in HBM, CUDA-graph
replay), timed in one process with CUDA events:

* ``train``: the training step (forward + ``loss.backward()``) with ``x.requires_grad`` False and True, alternating
  blocks on one model (both input geometries captured);
* ``attack``: one eval-mode attack iteration with every parameter frozen: forward + ``torch.autograd.grad(loss, x)``;
* ``cabinet_stem_dgrad`` alone over many launches, against its floors: bytes (dy of both stems + the fp32 dx) over the
  HBM data-sheet bandwidth, and the tensor-core work as issued (N = 4 parity classes x 3 channels padded to 16, K = 64
  per 7x7 view and 16 per 3x3 view) over the dense bf16 data-sheet rate.  dy (335 MB) is larger than the 126 MB L2.

Prints one line per measurement, then one JSON line with the card's name and power limit.

    python tools/bench_input_grad.py [--steps 20] [--warmup 5] [--kernel-iters 200]
"""

import argparse
import json
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

import torch  # noqa: E402

from cabinet_b200 import _lib  # noqa: E402
from cabinet_b200._lib import BF16, check  # noqa: E402
from cabinet_b200.loss import OhemCELoss  # noqa: E402
from cabinet_b200.synthetic import build_model, make_input, make_labels  # noqa: E402
from tools.bench_freeze import card  # noqa: E402

HBM_BYTES_PER_S = 7.7e12      # HGX B200 data sheet, one GPU
BF16_FLOP_PER_S = 2.25e15     # dense bf16, the same data sheet


def stem_dgrad_floors(N, H, W):
    """-> (bytes, issued MMA flops) of one cabinet_stem_dgrad call with bf16 dy."""
    OH, OW = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    nbytes = N * OH * OW * (64 + 16) * 2 + N * 3 * H * W * 4
    strips = -(-((W + 1) // 2) // 128)
    # per 128-column tile of a class row: 16 dy views of the 7x7 stem (K = 64) and 4 of the 3x3 stem (K = 16), N = 16
    flops = 2 * N * OH * strips * 128 * 16 * (16 * 64 + 4 * 16)
    return nbytes, flops


def timed(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--kernel-iters", type=int, default=200)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--size", type=int, default=1024)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    assert args.steps >= 10 and args.warmup >= 3, "time >= 10 steps after >= 3 warm-up steps (graph capture at step 3)"
    B, H, W, C = args.batch, args.size, args.size, 8
    x, lb = make_input(B, H, W, seed=7).cuda(), make_labels(B, H, W, C, seed=11).cuda()
    crit = OhemCELoss(0.7, B * H * W // 16, 255)
    rows = []

    # ---- the training step, with and without the input gradient
    model = build_model(C, "large").cuda().train()
    model.train_precision = "bf16"
    xg = x.clone().requires_grad_(True)

    def train_step(inp):
        def run():
            model.zero_grad(set_to_none=False)
            inp.grad = None
            out, out16 = model(inp)
            loss = crit(out, lb) + crit(out16, lb)
            loss.backward()
            return loss.detach()
        return run

    for inp in (x, xg):
        for _ in range(args.warmup):
            train_step(inp)()
    torch.cuda.synchronize()
    for rnd in range(2):
        for name, inp in (("train", x), ("train_input_grad", xg)):
            ms, loss = timed(train_step(inp), args.steps)
            rows.append({"round": rnd, "what": name, "ms": round(ms, 3), "img_per_s": round(B / ms * 1e3, 1)})
            print(f"round {rnd} {name:>17}: {ms:.3f} ms/step  {B / ms * 1e3:.1f} img/s  (loss {float(loss):.5f})", flush=True)
    del model, xg

    # ---- one eval-mode attack iteration, parameters frozen
    victim = build_model(C, "large").cuda().eval()
    victim.train_precision = "bf16"
    for p in victim.parameters():
        p.requires_grad_(False)

    def attack():
        xa = x.clone().requires_grad_(True)
        out, out16 = victim(xa)
        (g,) = torch.autograd.grad(crit(out, lb) + crit(out16, lb), xa)
        return g

    for _ in range(args.warmup):
        attack()
    torch.cuda.synchronize()
    for rnd in range(2):
        ms, _ = timed(attack, args.steps)
        rows.append({"round": rnd, "what": "attack_iteration", "ms": round(ms, 3), "img_per_s": round(B / ms * 1e3, 1)})
        print(f"round {rnd}  attack iteration: {ms:.3f} ms  {B / ms * 1e3:.1f} img/s", flush=True)
    del victim

    # ---- the kernel alone
    lib = _lib.load()
    OH, OW = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    g = torch.Generator(device="cuda").manual_seed(3)
    dy7 = torch.randn(B, OH, OW, 64, device="cuda", generator=g).to(torch.bfloat16)
    dy3 = torch.randn(B, OH, OW, 16, device="cuda", generator=g).to(torch.bfloat16)
    w7 = torch.randn(64, 3, 7, 7, device="cuda", generator=g) * 0.1
    w3 = torch.randn(16, 3, 3, 3, device="cuda", generator=g) * 0.3
    dx = torch.empty(B, 3, H, W, device="cuda")
    st = torch.cuda.current_stream().cuda_stream

    def kernel():
        check(lib.cabinet_stem_dgrad(dy7.data_ptr(), 64, dy3.data_ptr(), 16, BF16, w7.data_ptr(), w3.data_ptr(), dx.data_ptr(),
                                     B, H, W, OH, OW, st), "stem_dgrad")

    for _ in range(10):
        kernel()
    torch.cuda.synchronize()
    nbytes, flops = stem_dgrad_floors(B, H, W)
    byte_floor_us, mma_floor_us = nbytes / HBM_BYTES_PER_S * 1e6, flops / BF16_FLOP_PER_S * 1e6
    for rnd in range(2):
        ms, _ = timed(kernel, args.kernel_iters)
        us = ms * 1e3
        bound = "bytes" if byte_floor_us >= mma_floor_us else "MMA"
        rows.append({"round": rnd, "what": "cabinet_stem_dgrad", "us": round(us, 2), "byte_floor_us": round(byte_floor_us, 2),
                     "mma_floor_us": round(mma_floor_us, 2), "bound_by": bound,
                     "share_of_floor": round(max(byte_floor_us, mma_floor_us) / us, 3)})
        print(f"round {rnd} cabinet_stem_dgrad: {us:.1f} us  ({nbytes / 1e6:.0f} MB -> byte floor {byte_floor_us:.1f} us; "
              f"{flops / 1e9:.0f} GFLOP issued -> MMA floor {mma_floor_us:.1f} us; the {bound} floor bounds it, "
              f"{max(byte_floor_us, mma_floor_us) / us:.0%} of it)", flush=True)
    print(json.dumps({"card": card(), "workload": f"config 5: Large, batch {B}, {H}x{W}, {C} classes, bf16, graph replay",
                      "rows": rows}))


if __name__ == "__main__":
    main()
