"""Time a standalone MobileNetV3 against eager PyTorch of the same backbone on the same GPU, and its stem kernels.

    python tools/bench_backbone.py [--batch 16] [--hw 1024 1024] [--iters 20] [--warmup 5]

For Large and Small at batch 16, 1024 x 1024 (fp32 NCHW input, 201 MB: larger than the L2): the eval forward
(``precision='bf16'``) and the train forward + backward (``train_precision='bf16'``) of the drop-in, and eager PyTorch of
the reference backbone (``oracle.cabinet_oracle.mobilenet`` with fp32 weights under ``torch.autocast(bf16)``,
channels_last input and weights, cuDNN benchmark on).  The standalone backbone runs eagerly (no graph replay), so each
of its rows also gives the host's enqueue time per call (host clock from a synchronised start to the return of the
call) beside the device time.  The stem alone: ``cabinet_stem3_tc`` against ``cabinet_conv2d_simt`` on the same input,
with the bytes the layer has to move (fp32 input read once, bf16 16-channel output written once) over the kernel time.
CUDA events around ``--iters`` calls after ``--warmup`` calls; prints the card name and power limit.
"""

from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

import torch  # noqa: E402

from cabinet_b200 import MobileNetV3  # noqa: E402
from cabinet_b200._lib import check  # noqa: E402
from cabinet_b200.constants import BACKBONE_CFGS  # noqa: E402
from cabinet_b200.synthetic import build_model  # noqa: E402
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


def enqueue_ms(fn, iters):
    """Host time from a synchronised start to the return of ``fn`` (the kernels are queued, not finished)."""
    total = 0.0
    for _ in range(iters):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        total += time.perf_counter() - t0
    torch.cuda.synchronize()
    return 1e3 * total / iters


def make_backbone(mode):
    mob = MobileNetV3(BACKBONE_CFGS[mode], mode, num_classes=5)
    mob.load_state_dict(build_model(5, mode).mobile.state_dict())
    return mob.cuda()


def stem_rows(mob, x, iters, warmup):
    """cabinet_stem3_tc against cabinet_conv2d_simt (the engine's two routes for the stem) on the same input."""
    mob.eval()
    mob.precision = "bf16"
    eng = mob.engine()
    N, _, H, W = x.shape
    OH, OW = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    y_tc = eng.new(N, OH, OW, 16)

    def tc():
        check(eng.lib.cabinet_stem3_tc(x.data_ptr(), N, H, W, eng.stem_tc3.data_ptr(), y_tc.ptr, y_tc.ld, OH, OW,
                                       eng.stream), "stem3_tc")

    box = {}

    def simt():
        box["y"] = eng.conv(None, eng.stem, nchw_input=x)

    t_tc, t_simt = timed(tc, iters, warmup), timed(simt, iters, warmup)
    t_tc2, t_simt2 = timed(tc, iters, warmup), timed(simt, iters, warmup)   # alternated: two samples each
    diff = (y_tc.t.float() - box["y"].t.float()).norm() / box["y"].t.float().norm()
    nbytes = x.numel() * 4 + N * OH * OW * 16 * 2
    return [dict(kernel=k, batch=N, hw=f"{H}x{W}", ms=[round(a, 4), round(b, 4)], bytes=nbytes,
                 tb_per_s=round(nbytes / (min(a, b) * 1e-3) / 1e12, 2))
            for k, a, b in (("cabinet_stem3_tc", t_tc, t_tc2), ("cabinet_conv2d_simt", t_simt, t_simt2))], float(diff)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--hw", type=int, nargs=2, default=(1024, 1024))
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    a = ap.parse_args()
    torch.backends.cudnn.benchmark = True
    H, W = a.hw
    x = torch.randn(a.batch, 3, H, W, device="cuda", generator=torch.Generator("cuda").manual_seed(0))
    x_cl = x.contiguous(memory_format=torch.channels_last)
    rows, stems, stem_diff = [], None, None
    for mode in ("large", "small"):
        mob = make_backbone(mode)
        if stems is None:
            stems, stem_diff = stem_rows(mob, x, 5 * a.iters, a.warmup)
        sd = {"m." + k: (v.contiguous(memory_format=torch.channels_last) if v.dim() == 4 else v)
              for k, v in mob.state_dict().items()}
        params = {k: v.detach().clone().requires_grad_(True) for k, v in sd.items()
                  if not k.endswith(("running_mean", "running_var", "num_batches_tracked")) and ".classifier." not in k}
        work = dict(sd)
        work.update(params)
        cfgs = BACKBONE_CFGS[mode]

        mob.eval()
        mob.precision = "bf16"

        def ours_eval():
            with torch.no_grad():
                mob(x)

        t_eval = timed(ours_eval, a.iters, a.warmup)
        h_eval = enqueue_ms(ours_eval, a.iters)
        launches_eval = mob.engine().launches

        def ref_eval():
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
                cabinet_oracle.mobilenet(sd, x_cl, cfgs, p="m")

        t_ref_eval = timed(ref_eval, a.iters, a.warmup)

        mob.train()
        mob.train_precision = "bf16"
        with torch.no_grad():
            w = torch.randn_like(mob(x))

        def ours_step():
            (mob(x) * w).sum().backward()

        t_train = timed(ours_step, a.iters, a.warmup)
        h_train = enqueue_ms(ours_step, a.iters)

        def ref_step():
            cabinet_oracle.BATCH_STATS = {}
            try:
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    y = cabinet_oracle.mobilenet(work, x_cl, cfgs, p="m")
                (y.float() * w).sum().backward()
            finally:
                cabinet_oracle.BATCH_STATS = None

        t_ref_train = timed(ref_step, a.iters, a.warmup)
        rows.append(dict(backbone=f"MobileNetV3-{mode.capitalize()}", batch=a.batch, hw=f"{H}x{W}",
                         eval_ms=round(t_eval, 3), eval_host_enqueue_ms=round(h_eval, 3), eval_launches=launches_eval,
                         eval_torch_bf16_autocast_ms=round(t_ref_eval, 3), train_ms=round(t_train, 3),
                         train_host_enqueue_ms=round(h_train, 3), train_torch_bf16_autocast_ms=round(t_ref_train, 3)))
        del mob, sd, params, work
        torch.cuda.empty_cache()
    print(json.dumps(dict(card=card(), rows=rows, stem=stems, stem_rel_diff_tc_vs_simt=stem_diff), indent=1))


if __name__ == "__main__":
    main()
