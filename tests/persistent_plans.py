"""Host tile plans of the persistent inference kernels, and the GPU cases that walk them past their first tile.

Each persistent kernel launches ``min(tiles, SMs)`` CTAs (``2 x SMs`` for ``mbconv_fused``, ``SMs / chunks`` per
channel chunk for ``expand_sums``) and every CTA then works through tiles ``blockIdx.x, + gridDim.x, ...``.  The second
and later tiles of a CTA run code its first tile never reaches: ring wrap-around and mbarrier phase flips, the A2 / D2
double buffers, the deferred project epilogue of ``mbconv_t``, the division-free tile walk, re-streamed weight chunks,
the second epilogue warpgroup of ``conv_tc``, and several CTAs adding into one pooling accumulator.

``plan(entry, a)`` mirrors the host code of each entry point (``launch_mt``, ``launch_mb``, ``cabinet_stem_tc2``,
``cabinet_expand_sums``, ``conv_tc_impl``) for one call given as ``{argument name: value}``.  Its ``key`` holds what the
kernel's code path depends on, plus the ragged last tile row / column; ``tiles``, ``grid`` and ``per_cta`` say how far
the walk goes.  ``production()`` records the bf16 forward and mask schedules of bench configs 2-4 at batch 1 with the
recording C-ABI double and scales each call to the bench batch.  ``CASES`` is one GPU case per production key
(``tests/test_gpu_persistent.py``), at the production H x W and a batch that gives every CTA several tiles.
"""

from __future__ import annotations

import re
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
HEADER = ROOT / "include" / "cabinet_b200.h"
SMS = 148  # B200

# bench.py CONFIGS 2-4: mode, H, W, batch per GPU, classes
BENCH = {2: ("large", 1024, 1024, 16, 8), 3: ("large", 1024, 2048, 8, 19), 4: ("small", 2160, 3840, 4, 8)}
ENTRIES = ("mbconv_t", "mbconv_fused", "stem_tc2", "expand_sums", "conv_tc_se", "conv_tc_imgw", "conv_tc_split_act")


def _arg_names():
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    out = {}
    for e in ENTRIES:
        m = re.search(r"\bcabinet_%s\s*\(([^)]*)\)" % e, text)
        out[e] = [re.split(r"[\s*]+", a.strip())[-1] for a in m.group(1).split(",")]
    return out


ARG_NAMES = _arg_names()


def _cdiv(a, b):
    return -(-a // b)


def _walk(tiles, grid, tail_tiles):
    """per-CTA tile count, whether the last wave is partial, and whether a ragged tile is some CTA's 2nd+ tile."""
    return dict(tiles=tiles, grid=grid, per_cta=tiles / grid, partial_wave=tiles % grid != 0,
                tail_late=any(t >= grid for t in tail_tiles))


def _tail_tiles(N, tiles_w, tiles_h, tail_r, tail_c, per_tile=1):
    """linear tile indices (image-major, then row, then column) of the ragged tiles of the last image."""
    base = (N - 1) * tiles_w * tiles_h
    out = []
    if tail_r:
        out += [base + (tiles_h - 1) * tiles_w + c for c in range(tiles_w)]
    if tail_c:
        out += [base + r * tiles_w + tiles_w - 1 for r in range(tiles_h)]
    return [t * per_tile + j for t in out for j in range(per_tile)]


def mt_geometry(k, s, project, cexp, cout, cin):
    """launch_mt (mbconv_t.cu): template arguments, TMEM and shared-memory plan.  None = outside its budget (the engine
    then falls back to mbconv_fused)."""
    rep = 2 if cexp <= 64 else 1
    tw = {(3, 1): 16, (3, 2): 8, (5, 1): 8 if project else 16, (5, 2): 8}[(k, s)]
    th = 8 if s == 1 else 4
    nc = 1 if rep == 2 else _cdiv(cexp, 128)
    iwt, iht = (tw - 1) * s + k, (th - 1) * s + k
    ncols = _cdiv(iwt * iht, 16) * 16
    cout_pad = _cdiv(cout, 16) * 16 if project else 0
    d2_stride = _cdiv(cout_pad, 32) * 32
    nd2 = 2 if project and 2 * ncols + 2 * d2_stride <= 512 else 1
    d2col = 512 - nd2 * d2_stride if project else 512
    nd = min(4, d2col // ncols)
    if ncols > 256 or nd < 2:
        return None
    kb = cin // 64 + 1
    a1_stage = kb * _cdiv(ncols * 128, 1024) * 1024
    w1_buf, w2_buf = kb * 128 * 128, ((128 // rep) // 64) * cout_pad * 128 if project else 0
    resident = nc <= 2
    nw2 = 2
    fixed = 2 * w1_buf + 2 * w2_buf + (2 * 2 * 128 * 128 if project else 0) + 1024 + cout_pad * 4 + 1024
    if project and not resident and (226 * 1024 - fixed) // a1_stage < 2:
        nw2, fixed = 1, fixed - w2_buf
    ns = min(4, (226 * 1024 - fixed) // a1_stage)
    if ns < 1:
        return None
    return dict(rep=rep, TW=tw, TH=th, nc=nc, resident=resident, nd2=nd2, nw2=nw2, ns=ns, nd=nd)


def mb_geometry(k, s, project, cexp, cout, cin):
    """launch_mb (mbconv_fused.cu): the tile shape its shared-memory / TMEM probe picks."""
    cands = {(3, 1): [(8, 16), (8, 8)], (5, 1): [(8, 16), (8, 8)], (3, 2): [(4, 16), (4, 8)], (5, 2): [(4, 8)]}[(k, s)]
    nch = _cdiv(cexp, 64)
    kb = cin // 64 + 1
    cout_pad = _cdiv(cout, 16) * 16 if project else 0
    for th, tw in cands:
        npix = ((tw - 1) * s + k) * ((th - 1) * s + k)
        if _cdiv(npix, 128) * 64 + cout_pad > 256:
            continue
        e = _cdiv(npix * 144, 1024) * 1024
        if project and cout_pad > 64:
            e = max(e, (_cdiv(cout_pad, 64) - 1) * 128 * 128)
        if not project:
            e = max(e, _cdiv(128 * 144, 1024) * 1024)
        off_a2 = kb * _cdiv(npix * 128, 1024) * 1024 + e
        off_w = off_a2 + _cdiv(th * tw * 128, 1024) * 1024
        w_buf = _cdiv(kb * 64 * 128 + cout_pad * 128 + (k * k + 2) * 256, 1024) * 1024
        if max(off_w + min(nch, 2) * w_buf, off_a2 + 128 * 128) + cout_pad * 4 + 1024 <= 113 * 1024:
            return dict(TW=tw, TH=th, nc=nch, resident=nch <= 2)
    return None


def _spatial(entry, N, OH, OW, TH, TW, grid_cap, extra, per_tile=1):
    tiles_w, tiles_h = _cdiv(OW, TW), _cdiv(OH, TH)
    tail_r, tail_c = OH % TH, OW % TW
    tiles = N * tiles_w * tiles_h * per_tile
    grid = min(tiles, grid_cap)
    key = (entry,) + extra + (f"{TH}x{TW}", f"tail{tail_r},{tail_c}")
    return dict(key=key, TH=TH, TW=TW, tail=(tail_r, tail_c), tiles_img=tiles_w * tiles_h * per_tile,
                **_walk(tiles, grid, _tail_tiles(N, tiles_w, tiles_h, tail_r, tail_c, per_tile)))


def plan(entry, a, sms=SMS):
    """Host plan of one call ({argument name: value}); None = the entry point refuses it for its budget."""
    N = a["N"]
    if entry == "mbconv_t":
        project = bool(a["w_project"])
        mode = "se" if a["se_scale"] else ("project" if project else "dw+sums")
        g = mt_geometry(a["k"], a["stride"], project, a["Cexp"], a["Cout"], a["Cin"])
        if g is None:
            return None
        extra = (mode, f"k{a['k']}s{a['stride']}", f"rep{g['rep']}", f"nc{g['nc']}", "res" if g["resident"] else "stream",
                 f"nd2={g['nd2']}", f"nw2={g['nw2']}", f"ns{g['ns']}", f"nd{g['nd']}", "id" if a["residual"] else "")
        p = _spatial(entry, N, a["OH"], a["OW"], g["TH"], g["TW"], sms, extra)
    elif entry == "mbconv_fused":
        project = bool(a["w_project"])
        g = mb_geometry(a["k"], a["stride"], project, a["Cexp"], a["Cout"], a["Cin"])
        if g is None:
            return None
        extra = ("project" if project else "dw+sums", f"k{a['k']}s{a['stride']}", f"nc{g['nc']}",
                 "res" if g["resident"] else "stream", "id" if a["residual"] else "")
        p = _spatial(entry, N, a["OH"], a["OW"], g["TH"], g["TW"], 2 * sms, extra)
        # the tile shape comes from a probe of the kernel's budget: every shape it could pick must meet the same bar
        k, s = a["k"], a["stride"]
        alts = [(th, tw) for th, tw in ([(8, 16), (8, 8)] if s == 1 else ([(4, 16), (4, 8)] if k == 3 else [(4, 8)]))]
        p["alt_walks"] = [_spatial(entry, N, a["OH"], a["OW"], th, tw, 2 * sms, extra) for th, tw in alts]
    elif entry == "stem_tc2":
        p = _spatial(entry, N, a["OH"], a["OW"], 16, 8, sms, ())
    elif entry == "expand_sums":
        k, H, W, cexp = a["k"], a["H"], a["W"], a["Cexp"]
        rpb = max(1, 256 // W)
        nblk = _cdiv(H, rpb)
        nc = _cdiv(cexp, 128)
        cpc = max(1, sms // nc)
        nsplit = a["nsplit"] if a["nsplit"] > 0 else max(1, min(nblk, (2 * cpc + N - 1) // N - 1))
        units = N * (nsplit + 1)
        p = dict(key=(entry, f"k{k}", f"kb{a['Cin'] // 64 + 1}", f"nc{nc}", f"rpb{rpb}", f"nblk{nblk}", f"nsplit{nsplit}",
                      f"units{units}", f"cpc{cpc}"), nsplit=nsplit, tiles_img=nsplit + 1,
                 **_walk(units, min(cpc, units), []))
    else:  # conv_tc_impl: conv_tc_se / conv_tc_imgw / conv_tc_split_act
        KH, KW, s, Cin, Cout = a["KH"], a["KW"], a["stride"], a["Cin"], a["Cout"]
        flat = KH == 1 and KW == 1 and s == 1 and a["pad"] == 0
        n16 = _cdiv(Cout, 16) * 16
        n_tiles = _cdiv(n16, 256)
        block_n = n16 if n_tiles == 1 else 256
        b_res = entry != "conv_tc_imgw" and n_tiles == 1 and KH * KW * _cdiv(Cin, 64) * block_n * 128 <= 80 * 1024
        y_f32 = a["y_dtype"] == 0
        act = a["act"] & ~0x100
        extra = ("flat" if flat else f"k{KH}x{KW}s{s}", f"n{block_n}x{n_tiles}", "bres" if b_res else "bstream",
                 f"cbufs{2 if not y_f32 and block_n > 64 else 1}", "f32" if y_f32 else "bf16",
                 "res" if a.get("res") else "", "scale" if a.get("a_scale") else "", f"act{act}",
                 f"split{a['act_cols']}" if entry == "conv_tc_split_act" else "")
        if flat:
            P = N * a["H"] * a["W"]
            tiles_w = _cdiv(P, 128)
            tiles = tiles_w * n_tiles
            grid = min(tiles, sms)
            tail = P % 128
            p = dict(key=(entry,) + extra + ("128x1", f"tail0,{tail}"), TH=1, TW=128, tail=(0, tail),
                     tiles_img=a["H"] * a["W"] / 128 * n_tiles,
                     **_walk(tiles, grid, [(tiles_w - 1) * n_tiles + j for j in range(n_tiles)] if tail else []))
        else:
            best = None
            tw = 128
            while tw >= 4:
                th = 128 // tw
                cover = _cdiv(a["OW"], tw) * tw * _cdiv(a["OH"], th) * th
                if best is None or cover < best[0]:
                    best = (cover, tw, th)
                tw //= 2
            p = _spatial(entry, N, a["OH"], a["OW"], best[2], best[1], sms, extra, per_tile=n_tiles)
        # the second epilogue warpgroup takes tiles blockIdx.x + gridDim.x, + 3 gridDim.x, ...
        p["second_epilogue"] = p["tiles"] > p["grid"]
    p["entry"] = entry
    return p


def named(name, args):
    """recorded ``cabinet_X`` call -> (X, {argument name: value}); pointers are kept only as set / None."""
    entry = name[len("cabinet_"):]
    names = ARG_NAMES[entry]
    assert len(names) == len(args), (name, len(names), len(args))
    return entry, {n: (v if isinstance(v, int) or v is None else 1) for n, v in zip(names, args)}


def record(mode, H, W, classes):
    """(function, name, args) of every ABI call of the bf16 forward and forward_mask at batch 1 (no device needed)."""
    import torch

    from cabinet_b200 import _lib
    from cabinet_b200 import engine as engine_mod
    from cabinet_b200.synthetic import build_model
    from tests.test_engine_dryrun import RecordingLib

    class P:  # parameters that claim to live on a CUDA device
        is_cuda = True
        device = torch.device("cpu")

    rec = RecordingLib()
    saved_load, saved_stream = _lib.load, engine_mod.Engine.__dict__["stream"]
    _lib.load = lambda: rec
    engine_mod.Engine.stream = property(lambda self: None)
    try:
        engine_mod.next = lambda it: P
        try:
            eng = engine_mod.Engine(build_model(classes, mode), "bf16")
        finally:
            del engine_mod.next
        out = []
        x = torch.zeros(1, 3, H, W)
        for fn in ("forward", "forward_mask"):
            rec.calls.clear()
            getattr(eng, fn)(x)
            out += [(fn, n, a) for n, a in rec.calls]
        return out
    finally:
        _lib.load = saved_load
        engine_mod.Engine.stream = saved_stream


def production():
    """[(config, function, entry, args at the bench batch, plan)] for every persistent launch of configs 2-4."""
    out = []
    for cfg, (mode, H, W, B, C) in BENCH.items():
        for fn, name, args in record(mode, H, W, C):
            entry = name[len("cabinet_"):]
            if entry not in ENTRIES:
                continue
            entry, a = named(name, args)
            assert a["N"] == 1
            a["N"] = B
            p = plan(entry, a)
            assert p is not None, (cfg, entry, a)  # no recorded launch may be one the kernel refuses for its budget
            out.append((cfg, fn, entry, a, p))
    return out


def _case(entry, cfg, **a):
    """One GPU case; its id names the entry point, the bench config its geometry comes from, the shapes and the batch."""
    if entry in ("mbconv_t", "mbconv_fused"):
        mode = "se" if a.get("se_scale") else ("project" if a["w_project"] else "dw")
        shape = f"{a['Cin']}-{a['Cexp']}-{a['Cout']}-k{a['k']}s{a['stride']}-{mode}"
    elif entry == "stem_tc2":
        shape = "stems"
    elif entry == "expand_sums":
        shape = f"{a['Cin']}-{a['Cexp']}-k{a['k']}"
    else:
        shape = f"{a['Cin']}-{a['Cout']}-k{a['KH']}s{a['stride']}" + ("-scale" if a.get("a_scale") else "") + \
            ("-res" if a.get("res") else "") + ("-f32" if a["y_dtype"] == 0 else "")
    return dict(id=f"{entry}-c{cfg}-{shape}-{a['H']}x{a['W']}-N{a['N']}", entry=entry, cfg=cfg, **a)


def case_plan(c, sms=SMS):
    return plan(c["entry"], {k: v for k, v in c.items() if k not in ("id", "entry", "cfg")}, sms)


# One case per production plan key (generated from production(), checked by tests/test_persistent_plan_cpu.py): the
# production geometry at the smallest batch (>= 2, so that the batch can be compared with its images run alone) that
# gives every CTA min(4, production) tiles or more, leaves a partial last wave where production has one, and reaches the
# ragged tail as a CTA's second or later tile.
CASES = [
    _case('mbconv_t', 2, N=2, H=256, W=256, Cin=24, Cexp=72, Cout=24, k=3, stride=1, act_expand=1, act_dw=1, OH=256,
          OW=256, residual=1, w_project=1, se_scale=None, gap_sum=None),
    _case('mbconv_t', 2, N=2, H=256, W=256, Cin=24, Cexp=72, Cout=0, k=5, stride=2, act_expand=1, act_dw=1, OH=128,
          OW=128, residual=0, w_project=None, se_scale=None, gap_sum=1),
    _case('mbconv_t', 2, N=5, H=128, W=128, Cin=40, Cexp=120, Cout=0, k=5, stride=1, act_expand=1, act_dw=1, OH=128,
          OW=128, residual=0, w_project=None, se_scale=None, gap_sum=1),
    _case('mbconv_t', 2, N=5, H=128, W=128, Cin=40, Cexp=240, Cout=80, k=3, stride=2, act_expand=2, act_dw=2, OH=64,
          OW=64, residual=0, w_project=1, se_scale=None, gap_sum=None),
    _case('mbconv_t', 2, N=16, H=64, W=64, Cin=80, Cexp=200, Cout=80, k=3, stride=1, act_expand=2, act_dw=2, OH=64,
          OW=64, residual=1, w_project=1, se_scale=None, gap_sum=None),
    _case('mbconv_t', 2, N=16, H=64, W=64, Cin=80, Cexp=480, Cout=112, k=3, stride=1, act_expand=2, act_dw=2, OH=64,
          OW=64, residual=0, w_project=1, se_scale=1, gap_sum=None),
    _case('mbconv_t', 2, N=16, H=64, W=64, Cin=112, Cexp=672, Cout=112, k=3, stride=1, act_expand=2, act_dw=2, OH=64,
          OW=64, residual=1, w_project=1, se_scale=1, gap_sum=None),
    _case('mbconv_t', 2, N=16, H=64, W=64, Cin=112, Cexp=672, Cout=0, k=5, stride=2, act_expand=2, act_dw=0, OH=32,
          OW=32, residual=0, w_project=None, se_scale=None, gap_sum=1),
    _case('mbconv_t', 2, N=2, H=32, W=32, Cin=160, Cexp=960, Cout=0, k=5, stride=1, act_expand=2, act_dw=0, OH=32,
          OW=32, residual=0, w_project=None, se_scale=None, gap_sum=1),
    _case('mbconv_t', 4, N=2, H=540, W=960, Cin=16, Cexp=72, Cout=24, k=3, stride=2, act_expand=1, act_dw=1, OH=270,
          OW=480, residual=0, w_project=1, se_scale=None, gap_sum=None),
    _case('mbconv_t', 4, N=2, H=270, W=480, Cin=24, Cexp=88, Cout=24, k=3, stride=1, act_expand=1, act_dw=1, OH=270,
          OW=480, residual=1, w_project=1, se_scale=None, gap_sum=None),
    _case('mbconv_t', 4, N=2, H=270, W=480, Cin=24, Cexp=96, Cout=0, k=5, stride=2, act_expand=2, act_dw=0, OH=135,
          OW=240, residual=0, w_project=None, se_scale=None, gap_sum=1),
    _case('mbconv_t', 4, N=3, H=135, W=240, Cin=40, Cexp=240, Cout=0, k=5, stride=1, act_expand=2, act_dw=0, OH=135,
          OW=240, residual=0, w_project=None, se_scale=None, gap_sum=1),
    _case('mbconv_t', 4, N=3, H=135, W=240, Cin=40, Cexp=120, Cout=0, k=5, stride=1, act_expand=2, act_dw=0, OH=135,
          OW=240, residual=0, w_project=None, se_scale=None, gap_sum=1),
    _case('mbconv_t', 4, N=3, H=135, W=240, Cin=48, Cexp=288, Cout=0, k=5, stride=2, act_expand=2, act_dw=0, OH=68,
          OW=120, residual=0, w_project=None, se_scale=None, gap_sum=1),
    _case('mbconv_t', 4, N=4, H=68, W=120, Cin=96, Cexp=576, Cout=0, k=5, stride=1, act_expand=2, act_dw=0, OH=68,
          OW=120, residual=0, w_project=None, se_scale=None, gap_sum=1),
    _case('mbconv_fused', 2, N=2, H=512, W=512, Cin=16, Cexp=64, Cout=24, k=3, stride=2, act_expand=1, act_dw=1, OH=256,
          OW=256, residual=0, w_project=1, gap_sum=None),
    _case('stem_tc2', 2, N=2, H=1024, W=1024, OH=512, OW=512),
    _case('stem_tc2', 4, N=2, H=2160, W=3840, OH=1080, OW=1920),
    _case('expand_sums', 2, N=16, H=64, W=64, Cin=80, Cexp=480, act_expand=2, k=3, nsplit=0, gap_sum=1),
    _case('expand_sums', 2, N=16, H=64, W=64, Cin=112, Cexp=672, act_expand=2, k=3, nsplit=0, gap_sum=1),
    _case('expand_sums', 3, N=8, H=64, W=128, Cin=80, Cexp=480, act_expand=2, k=3, nsplit=0, gap_sum=1),
    _case('expand_sums', 3, N=8, H=64, W=128, Cin=112, Cexp=672, act_expand=2, k=3, nsplit=0, gap_sum=1),
    _case('conv_tc_se', 2, N=5, H=256, W=256, Cin=64, Cout=64, KH=3, KW=3, stride=2, pad=1, y_dtype=1, OH=128, OW=128,
          act=1, a_act=0, res=None, a_scale=None),
    _case('conv_tc_se', 2, N=5, H=128, W=128, Cin=64, Cout=128, KH=1, KW=1, stride=1, pad=0, y_dtype=1, OH=128, OW=128,
          act=1, a_act=0, res=None, a_scale=None),
    _case('conv_tc_se', 2, N=2, H=32, W=32, Cin=672, Cout=160, KH=1, KW=1, stride=1, pad=0, y_dtype=1, OH=32, OW=32,
          act=0, a_act=2, res=None, a_scale=1),
    _case('conv_tc_se', 2, N=2, H=32, W=32, Cin=960, Cout=160, KH=1, KW=1, stride=1, pad=0, y_dtype=1, OH=32, OW=32,
          act=0, a_act=0, res=1, a_scale=None),
    _case('conv_tc_se', 2, N=16, H=32, W=32, Cin=160, Cout=960, KH=1, KW=1, stride=1, pad=0, y_dtype=1, OH=32, OW=32,
          act=2, a_act=0, res=None, a_scale=None),
    _case('conv_tc_se', 2, N=2, H=32, W=32, Cin=960, Cout=256, KH=3, KW=3, stride=1, pad=1, y_dtype=1, OH=32, OW=32,
          act=1, a_act=0, res=None, a_scale=None),
    _case('conv_tc_se', 2, N=75, H=32, W=32, Cin=256, Cout=8, KH=1, KW=1, stride=1, pad=0, y_dtype=0, OH=32, OW=32,
          act=0, a_act=0, res=None, a_scale=None),
    _case('conv_tc_se', 2, N=5, H=128, W=128, Cin=384, Cout=256, KH=1, KW=1, stride=1, pad=0, y_dtype=1, OH=128, OW=128,
          act=1, a_act=0, res=None, a_scale=None),
    _case('conv_tc_se', 3, N=2, H=32, W=64, Cin=960, Cout=256, KH=3, KW=3, stride=1, pad=1, y_dtype=1, OH=32, OW=64,
          act=1, a_act=0, res=None, a_scale=None),
    _case('conv_tc_se', 3, N=38, H=32, W=64, Cin=256, Cout=19, KH=1, KW=1, stride=1, pad=0, y_dtype=0, OH=32, OW=64,
          act=0, a_act=0, res=None, a_scale=None),
    _case('conv_tc_se', 4, N=4, H=68, W=120, Cin=640, Cout=128, KH=1, KW=1, stride=1, pad=0, y_dtype=1, OH=68, OW=120,
          act=0, a_act=0, res=None, a_scale=None),
    _case('conv_tc_se', 4, N=4, H=68, W=120, Cin=128, Cout=256, KH=1, KW=1, stride=1, pad=0, y_dtype=1, OH=68, OW=120,
          act=0, a_act=0, res=None, a_scale=None),
    _case('conv_tc_se', 4, N=4, H=68, W=120, Cin=256, Cout=256, KH=1, KW=1, stride=1, pad=0, y_dtype=1, OH=68, OW=120,
          act=0, a_act=0, res=None, a_scale=None),
    _case('conv_tc_se', 4, N=2, H=1080, W=1920, Cin=64, Cout=64, KH=3, KW=3, stride=2, pad=1, y_dtype=1, OH=540, OW=960,
          act=1, a_act=0, res=None, a_scale=None),
    _case('conv_tc_se', 4, N=2, H=540, W=960, Cin=64, Cout=64, KH=3, KW=3, stride=2, pad=1, y_dtype=1, OH=270, OW=480,
          act=1, a_act=0, res=None, a_scale=None),
    _case('conv_tc_se', 4, N=2, H=540, W=960, Cin=16, Cout=16, KH=1, KW=1, stride=1, pad=0, y_dtype=1, OH=540, OW=960,
          act=0, a_act=0, res=None, a_scale=None),
    _case('conv_tc_se', 4, N=4, H=135, W=240, Cin=96, Cout=40, KH=1, KW=1, stride=1, pad=0, y_dtype=1, OH=135, OW=240,
          act=0, a_act=0, res=None, a_scale=None),
    _case('conv_tc_se', 4, N=4, H=135, W=240, Cin=240, Cout=40, KH=1, KW=1, stride=1, pad=0, y_dtype=1, OH=135, OW=240,
          act=0, a_act=0, res=1, a_scale=None),
    _case('conv_tc_se', 4, N=4, H=68, W=120, Cin=288, Cout=96, KH=1, KW=1, stride=1, pad=0, y_dtype=1, OH=68, OW=120,
          act=0, a_act=0, res=None, a_scale=None),
    _case('conv_tc_se', 4, N=4, H=68, W=120, Cin=576, Cout=96, KH=1, KW=1, stride=1, pad=0, y_dtype=1, OH=68, OW=120,
          act=0, a_act=0, res=1, a_scale=None),
    _case('conv_tc_se', 4, N=4, H=68, W=120, Cin=96, Cout=576, KH=1, KW=1, stride=1, pad=0, y_dtype=1, OH=68, OW=120,
          act=2, a_act=0, res=None, a_scale=None),
    _case('conv_tc_se', 4, N=4, H=68, W=120, Cin=576, Cout=256, KH=3, KW=3, stride=1, pad=1, y_dtype=1, OH=68, OW=120,
          act=1, a_act=0, res=None, a_scale=None),
    _case('conv_tc_imgw', 2, N=5, H=128, W=128, Cin=72, Cout=40, KH=1, KW=1, stride=1, pad=0, y_dtype=1, OH=128, OW=128,
          act=0, res=None),
    _case('conv_tc_imgw', 2, N=5, H=128, W=128, Cin=120, Cout=40, KH=1, KW=1, stride=1, pad=0, y_dtype=1, OH=128,
          OW=128, act=0, res=1),
    _case('conv_tc_imgw', 2, N=5, H=128, W=128, Cin=256, Cout=256, KH=3, KW=3, stride=1, pad=1, y_dtype=1, OH=128,
          OW=128, act=1, res=None),
    _case('conv_tc_imgw', 4, N=2, H=270, W=480, Cin=256, Cout=256, KH=3, KW=3, stride=1, pad=1, y_dtype=1, OH=270,
          OW=480, act=1, res=None),
    _case('conv_tc_split_act', 4, N=4, H=68, W=120, Cin=256, Cout=384, KH=1, KW=1, stride=1, pad=0, y_dtype=1, OH=68,
          OW=120, act=1, act_cols=256),
]
# the dominant launches at the full config-2 batch, and mbconv_fused in its depthwise-output mode (the forward's
# fall-back for the squeeze-excite blocks that mbconv_t cannot take)
CASES += [
    _case("stem_tc2", 2, N=16, H=1024, W=1024, OH=512, OW=512),
    _case("mbconv_t", 2, N=16, H=256, W=256, Cin=24, Cexp=72, Cout=24, k=3, stride=1, act_expand=1, act_dw=1, OH=256,
          OW=256, residual=1, w_project=1, se_scale=None, gap_sum=None),
    _case("mbconv_fused", 2, N=16, H=512, W=512, Cin=16, Cexp=64, Cout=24, k=3, stride=2, act_expand=1, act_dw=1,
          OH=256, OW=256, residual=0, w_project=1, gap_sum=None),
    _case("mbconv_fused", 2, N=2, H=512, W=512, Cin=16, Cexp=64, Cout=0, k=3, stride=2, act_expand=1, act_dw=1,
          OH=256, OW=256, residual=0, w_project=None, gap_sum=1),
]
