"""Time CABiNet's spatial branch, attention branch, fusion module and head on their own against eager PyTorch of the same
modules, and the sb.conv1-only stem kernel.

    python tools/bench_heads.py [--batch 16] [--hw 1024 1024] [--iters 20] [--warmup 5] [--out FILE]

CABiNet-Large shapes for a batch of 16 at 1024 x 1024: sb on 16 x 3 x 1024^2, ab on 16 x 960 x 32^2, ffm on
16 x (128 + 256) x 128^2, head on 16 x 256 x 128^2.  For each module: the eval forward (``precision='bf16'``) and the
train forward + backward (``train_precision='bf16'``) of the drop-in, and eager PyTorch of the oracle's function of the
same module (fp32 weights under ``torch.autocast(bf16)``, channels_last inputs and weights, cuDNN benchmark on).  The
modules run eagerly, so each row also gives the host's enqueue time per call beside the device time.  The stem alone:
``cabinet_stem7_tc`` against ``cabinet_conv2d_simt`` on the same layer and input, with the bytes the layer has to move
(fp32 input read once, bf16 64-channel output written once) over the kernel time, and the byte floor at the data sheet's
7.7 TB/s.  CUDA events around ``--iters`` calls after ``--warmup`` calls; prints the card name and power limit.
"""

from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

import torch  # noqa: E402

from cabinet_b200._lib import check  # noqa: E402
from cabinet_b200.synthetic import build_model  # noqa: E402
from oracle import cabinet_oracle  # noqa: E402
from tools.bench_backbone import card, enqueue_ms, timed  # noqa: E402

HBM_TB_S = 7.7   # HGX B200 data sheet, one GPU


def stem_rows(sb, x, iters, warmup):
    """cabinet_stem7_tc against cabinet_conv2d_simt (the engine's two routes for sb.conv1) on the same input."""
    sb.eval()
    sb.precision = "bf16"
    eng = sb.engine()
    N, _, H, W = x.shape
    OH, OW = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    y_tc = eng.new(N, OH, OW, 64)

    def tc():
        check(eng.lib.cabinet_stem7_tc(x.data_ptr(), N, H, W, eng.stem_tc7.data_ptr(), y_tc.ptr, y_tc.ld, OH, OW,
                                       eng.stream), "stem7_tc")

    box = {}

    def simt():
        box["y"] = eng.conv(None, eng.sb1, nchw_input=x)

    t_tc, t_simt = timed(tc, iters, warmup), timed(simt, iters, warmup)
    t_tc2, t_simt2 = timed(tc, iters, warmup), timed(simt, iters, warmup)   # alternated: two samples each
    diff = (y_tc.t.float() - box["y"].t.float()).norm() / box["y"].t.float().norm()
    nbytes = x.numel() * 4 + N * OH * OW * 64 * 2
    floor_ms = nbytes / (HBM_TB_S * 1e12) * 1e3
    return [dict(kernel=k, batch=N, hw=f"{H}x{W}", ms=[round(a, 4), round(b, 4)], bytes=nbytes,
                 tb_per_s=round(nbytes / (min(a, b) * 1e-3) / 1e12, 2),
                 byte_floor_ms_at_data_sheet=round(floor_ms, 4), floor_over_time=round(floor_ms / min(a, b), 3))
            for k, a, b in (("cabinet_stem7_tc", t_tc, t_tc2), ("cabinet_conv2d_simt", t_simt, t_simt2))], float(diff)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--hw", type=int, nargs=2, default=(1024, 1024))
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON here")
    a = ap.parse_args()
    torch.backends.cudnn.benchmark = True
    N, (H, W) = a.batch, a.hw
    g = torch.Generator("cuda").manual_seed(0)
    net = build_model(19, "large").cuda()
    h8, w8, h32, w32 = -(-H // 8), -(-W // 8), -(-H // 32), -(-W // 32)
    cases = {   # module, its inputs, the oracle's function of it (prefix "m.")
        "sb": (net.sb, [torch.randn(N, 3, H, W, device="cuda", generator=g)],
               lambda sd, xs: cabinet_oracle.spatial_branch(sd, xs[0], p="m")),
        "ab": (net.ab, [torch.randn(N, net.attention_planes, h32, w32, device="cuda", generator=g).relu()],
               lambda sd, xs: cabinet_oracle.attention_branch(sd, xs[0], p="m")),
        "ffm": (net.ffm, [torch.randn(N, 128, h8, w8, device="cuda", generator=g).relu(),
                          torch.randn(N, 256, h8, w8, device="cuda", generator=g)],
                lambda sd, xs: cabinet_oracle.ffm(sd, xs[0], xs[1], p="m")),
        "head": (net.conv_out, [torch.randn(N, 256, h8, w8, device="cuda", generator=g).relu()],
                 lambda sd, xs: cabinet_oracle.head(sd, xs[0], p="m")),
    }
    stems, stem_diff = stem_rows(net.sb, cases["sb"][1][0], 5 * a.iters, a.warmup)
    rows = []
    for name, (m, xs, ref) in cases.items():
        xs_cl = [x.contiguous(memory_format=torch.channels_last) for x in xs]
        sd = {"m." + k: (v.contiguous(memory_format=torch.channels_last) if v.dim() == 4 else v)
              for k, v in m.state_dict().items()}
        params = {k: v.detach().clone().requires_grad_(True) for k, v in sd.items()
                  if not k.endswith(("running_mean", "running_var", "num_batches_tracked"))}
        work = dict(sd)
        work.update(params)
        as_list = lambda y: list(y) if isinstance(y, tuple) else [y]  # noqa: E731

        m.eval()
        m.precision = "bf16"

        def ours_eval():
            with torch.no_grad():
                m(*xs)

        t_eval = timed(ours_eval, a.iters, a.warmup)
        h_eval = enqueue_ms(ours_eval, a.iters)
        launches_eval = m.engine().launches

        def ref_eval():
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
                ref(sd, xs_cl)

        t_ref_eval = timed(ref_eval, a.iters, a.warmup)

        m.train()
        m.train_precision = "bf16"
        with torch.no_grad():
            ws = [torch.randn_like(y) for y in as_list(m(*xs))]

        def ours_step():
            sum((y * w).sum() for y, w in zip(as_list(m(*xs)), ws)).backward()

        t_train = timed(ours_step, a.iters, a.warmup)
        h_train = enqueue_ms(ours_step, a.iters)

        def ref_step():
            cabinet_oracle.BATCH_STATS = {}
            try:
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    ys = as_list(ref(work, xs_cl))
                sum((y.float() * w).sum() for y, w in zip(ys, ws)).backward()
            finally:
                cabinet_oracle.BATCH_STATS = None

        t_ref_train = timed(ref_step, a.iters, a.warmup)
        rows.append(dict(module=name, inputs=[list(x.shape) for x in xs], eval_ms=round(t_eval, 3),
                         eval_host_enqueue_ms=round(h_eval, 3), eval_launches=launches_eval,
                         eval_torch_bf16_autocast_ms=round(t_ref_eval, 3), train_ms=round(t_train, 3),
                         train_host_enqueue_ms=round(h_train, 3), train_torch_bf16_autocast_ms=round(t_ref_train, 3)))
        m.eval()
        del sd, params, work
        torch.cuda.empty_cache()
    out = json.dumps(dict(card=card(), rows=rows, stem=stems, stem_rel_diff_tc_vs_simt=stem_diff), indent=1)
    print(out)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(out + "\n")


if __name__ == "__main__":
    main()
