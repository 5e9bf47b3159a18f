"""GPU: every variant of the training step's elementwise and reduction kernels that the step launches, replayed against
float64 references.

One case per variant key of ``tests/train_variants.py`` (the inputs of the host dispatch: types, channel windows,
alignment, vector-path conditions, the rt threshold, accumulate, act, NULL operands, resample flag bits), with the
geometry of a call recorded from the step (``tests/test_train_variants_cpu.py`` checks that the matrix covers every key
the step reaches).  For each case:

* every operand is a channel window of a wider buffer at the recorded pixel stride and base alignment; every byte outside
  the windows is a NaN canary and must be bit-unchanged after the call (a write into neighbouring concat channels or past
  the last pixel fails), and inputs must be bit-unchanged;
* the reference is computed in float64 from the same values rounded to the operand types; an accumulating output starts
  from known random values and is compared with ``prior + ref``;
* 2-byte outputs: elementwise within 2 ulp of the output type plus ``1e-6 * max|ref|`` of the float64 reference rounded
  to that type; fp32 outputs: rel-L2 < 1e-5, < 1e-4 where a sum runs over more than 1e5 rows;
* the call runs twice on the same inputs and must give bit-identical outputs (fixed-order reductions);
* BatchNorm cases that take the shared-memory-staged "rt" path run once more with bit 7 of ``cabinet_debug_flags`` (the
  register-fed path), against the same reference.
"""

import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from cabinet_b200 import _lib  # noqa: E402
from cabinet_b200._lib import F32, check  # noqa: E402
from cabinet_b200.train_engine import adaptive_pool_matrix, bilinear_matrix  # noqa: E402
from tests.train_variants import variant_key  # noqa: E402

TD = {0: torch.float32, 1: torch.bfloat16, 2: torch.float16}
ITD = {torch.float32: torch.int32, torch.bfloat16: torch.int16, torch.float16: torch.int16}
MANT = {torch.bfloat16: (7, -126), torch.float16: (10, -14)}   # mantissa bits, smallest normal exponent
LEAD = 64   # canary elements in front of every window (keeps 16-byte alignment for every element size)


def stream():
    return torch.cuda.current_stream().cuda_stream


def act_ref(u, act):
    return [lambda t: t, F.relu, F.hardswish, F.hardsigmoid, torch.sigmoid][act](u)


class Operand:
    """A [rows][C] window with pixel stride ld and base address = buffer + al bytes (mod 16) in a NaN-filled buffer."""

    def __init__(self, rows, C, ld, al, dtype, values, prior=None, out=False):
        self.dt = TD[dtype]
        es = self.dt.itemsize
        assert al % es == 0 and ld >= C
        off = al // es
        assert off + C <= ld or rows == 1, "a channel window at this alignment does not fit the pixel stride"
        self.rows, self.C, self.ld, self.out = rows, C, ld, out
        n = LEAD + off + (rows - 1) * ld + C + LEAD
        self.buf = torch.full((n,), float("nan"), dtype=self.dt, device="cuda")
        self.view = self.buf[LEAD + off:].as_strided((rows, C), (ld, 1))
        self.mask = torch.zeros(n, dtype=torch.bool, device="cuda")
        self.mask[LEAD + off:].as_strided((rows, C), (ld, 1)).fill_(True)
        self.ref = None if values is None else values.to(self.dt).double()   # the rounded values the kernel sees
        self.prior = None if prior is None else prior.to(self.dt).double()
        if values is not None:
            self.view.copy_(values.to(self.dt).cuda())
        self.snap = self.buf.clone()
        self.ptr = self.view.data_ptr()

    def reset(self):
        if self.out:
            if self.prior is not None:
                self.view.copy_(self.prior.to(self.dt).cuda())
            else:
                self.view.fill_(float("nan"))

    def check_canaries(self, what):
        keep = ~self.mask if self.out else torch.ones_like(self.mask)
        a, b = self.buf.view(ITD[self.dt])[keep], self.snap.view(ITD[self.dt])[keep]
        bad = (a != b).nonzero()
        assert bad.numel() == 0, f"{what}: {bad.numel()} bytes outside the output windows changed, first at element " \
                                 f"{int(bad[0]) - LEAD} of the buffer"

    def got(self):
        return self.view.double().cpu()


class Case:
    def __init__(self):
        self.ops, self.checks = [], []
        self.seed = 0

    def rnd(self, *shape, scale=1.0, shift=0.0):
        self.seed += 1
        return torch.randn(*shape, generator=torch.Generator().manual_seed(self.seed), dtype=torch.float64) * scale + shift

    def inp(self, rows, C, ld, al, dtype, values):
        op = Operand(rows, C, ld, al, dtype, values)
        self.ops.append(op)
        return op

    def vec(self, values, dtype=F32):   # a dense fp32 parameter / statistics vector
        v = values.reshape(1, -1)
        return self.inp(1, v.shape[1], v.shape[1], 0, dtype, v)

    def out(self, rows, C, ld, al, dtype, acc=False, prior=None):
        if acc and prior is None:
            prior = self.rnd(rows, C)
        op = Operand(rows, C, ld, al, dtype, None, prior if acc else None, out=True)
        self.ops.append(op)
        return op

    def expect(self, name, op, ref, tol=1e-5):
        """op (+ its prior when accumulating) must match the float64 reference ``ref`` [rows][C]."""
        self.checks.append((name, op, ref.reshape(op.rows, op.C) + (op.prior if op.prior is not None else 0), tol))


def ulp(r, dt):
    mant, emin = MANT[dt]
    e = torch.floor(torch.log2(r.abs().clamp_min(2.0 ** emin))).clamp_min(emin)
    return torch.pow(2.0, e - mant)


def compare(name, op, ref, tol):
    got = op.got()
    assert torch.isfinite(got).all(), f"{name}: {int((~torch.isfinite(got)).sum())} non-finite values"
    if op.dt == torch.float32:
        e = float((got - ref).norm() / ref.norm().clamp_min(1e-30))
        assert e < tol, f"{name}: rel_l2 {e:.3e} >= {tol:g}"
        return
    r = ref.to(op.dt).double()
    bound = 2 * ulp(r, op.dt) + 1e-6 * float(ref.abs().max())
    err = (got - r).abs()
    bad = (err > bound).nonzero()
    assert bad.numel() == 0, f"{name}: {bad.shape[0]} of {got.numel()} elements beyond 2 ulp, first {bad[0].tolist()}: " \
                             f"got {float(got[tuple(bad[0])])}, reference {float(ref[tuple(bad[0])])}"


def red_tol(rows):   # fp32 sums over more than 1e5 rows
    return 1e-4 if rows > 1e5 else 1e-5


def nchw(t, N, H, W):   # [N*H*W][C] -> [N][C][H][W]
    return t.reshape(N, H, W, -1).permute(0, 3, 1, 2)


def rows_of(t):   # [N][C][H][W] -> [N*H*W][C]
    return t.permute(0, 2, 3, 1).reshape(-1, t.shape[1])


def scratch(lib, M, C, nq):
    return torch.empty(max(int(lib.cabinet_train_scratch_floats(M, C, nq)), 1), device="cuda")


# ----------------------------------------------------------------------------------------------------------- runners
def bn_stats_for(k, z, C):   # fp32 stats[4][C] of the rounded map z [M][C] (mean >> std: the shifted sums must not cancel)
    gamma, beta = k.rnd(C, scale=0.3, shift=1.0), k.rnd(C, scale=0.2)
    mean, var = z.mean(0), z.var(0, unbiased=False)
    invstd = (var + 1e-5).rsqrt()
    scale = gamma * invstd
    return torch.stack([mean, invstd, scale, beta - mean * scale]).float().double()


def run_bn_train_stats(lib, a, k):
    M, C, dt = a["M"], a["C"], a["dtype"]
    x = k.inp(M, C, a["ldx"], a["x"], dt, k.rnd(M, C, scale=2.0, shift=5.0))
    gamma, beta = k.vec(k.rnd(C, scale=0.3, shift=1.0)), k.vec(k.rnd(C, scale=0.2))
    rm = k.out(1, C, C, 0, F32, acc=True, prior=k.rnd(1, C, scale=0.1))
    rv = k.out(1, C, C, 0, F32, acc=True, prior=k.rnd(1, C).abs() + 0.5)
    stats = k.out(4, C, C, 0, F32)
    sc = scratch(lib, M, C, 2)
    eps, mom = a["eps"], a["momentum"]
    xr = x.ref
    mean, var = xr.mean(0), xr.var(0, unbiased=False)
    invstd = (var + eps).rsqrt()
    scale = gamma.ref[0] * invstd
    ref = torch.stack([mean, invstd, scale, beta.ref[0] - mean * scale])
    for i, nm in enumerate(("mean", "invstd", "scale", "shift")):
        k.checks.append((f"stats.{nm}", _Row(stats, i), ref[i:i + 1], red_tol(M)))
    k.expect("running_mean", rm, mom * mean - mom * rm.prior[0], red_tol(M))
    k.expect("running_var", rv, mom * var * M / (M - 1) - mom * rv.prior[0], red_tol(M))
    return lambda: lib.cabinet_bn_train_stats(x.ptr, a["ldx"], dt, M, C, gamma.ptr, beta.ptr, eps, mom, rm.ptr, rv.ptr,
                                              stats.ptr, sc.data_ptr(), stream())


class _Row:   # one row of an output operand, compared on its own
    def __init__(self, op, i):
        self.op, self.i, self.rows, self.C, self.dt, self.prior = op, i, 1, op.C, op.dt, None

    def got(self):
        return self.op.got()[self.i:self.i + 1]


def _bn_backward(lib, a, k, frozen):
    M, C, dt, act = a["M"], a["C"], a["dtype"], a["act"]
    z = k.inp(M, C, a["ldz"], a["z"], dt, k.rnd(M, C, scale=2.0, shift=5.0))
    dy = k.inp(M, C, a["lddy"], a["dy"], dt, k.rnd(M, C))
    st = bn_stats_for(k, z.ref, C)
    if frozen:   # eval-mode statistics: running mean / variance away from the batch's
        st[0] += k.rnd(C, scale=0.5)
        st[1] *= 1.0 + 0.3 * torch.rand(C, generator=torch.Generator().manual_seed(7), dtype=torch.float64)
        st[3] = -st[0] * st[2] + k.rnd(C, scale=0.2)
        st = st.float().double()
    stats = k.inp(4, C, C, 0, F32, st)
    dz = k.out(M, C, a["lddz"], a["dz"], dt, acc=a["accumulate"]) if a["dz"] is not None else None
    dgamma = k.out(1, C, C, 0, F32, acc=True) if a["dgamma"] is not None else None
    dbeta = k.out(1, C, C, 0, F32, acc=True) if a["dbeta"] is not None else None
    sc = scratch(lib, M, C, 2 if frozen else 4)
    mean, invstd, scale, shift = stats.ref
    u = (z.ref * scale + shift).requires_grad_(True)
    act_ref(u, act).backward(dy.ref)
    g = u.grad
    xhat = (z.ref - mean) * invstd
    if dbeta is not None:
        k.expect("dbeta", dbeta, g.sum(0), red_tol(M))
    if dgamma is not None:
        k.expect("dgamma", dgamma, (g * xhat).sum(0), red_tol(M))
    if dz is not None:
        k.expect("dz", dz, scale * g if frozen else scale * (g - g.mean(0) - xhat * (g * xhat).mean(0)), red_tol(M))
    fn = lib.cabinet_bn_frozen_backward if frozen else lib.cabinet_bn_train_backward
    p = lambda o: None if o is None else o.ptr  # noqa: E731
    return lambda: fn(dy.ptr, a["lddy"], z.ptr, a["ldz"], dt, stats.ptr, act, p(dgamma), p(dbeta), p(dz),
                      a["lddz"], M, C, a["accumulate"], sc.data_ptr(), stream())


def run_bn_train_backward(lib, a, k):
    return _bn_backward(lib, a, k, False)


def run_bn_frozen_backward(lib, a, k):
    return _bn_backward(lib, a, k, True)


def run_affine_act(lib, a, k):
    M, HW, C, act = a["M"], a["HW"], a["C"], a["act"]
    N = M // HW
    z = k.inp(M, C, a["ldz"], a["z"], a["z_dtype"], k.rnd(M, C, scale=2.0))
    u = z.ref
    scale = shift = gate = res = None
    if a["scale"] is not None:
        scale, shift = k.vec(k.rnd(C, scale=0.5, shift=1.0)), k.vec(k.rnd(C, scale=0.5))
        u = u * scale.ref + shift.ref
    if a["gate"] is not None:
        gate = k.inp(N, C, C, 0, F32, torch.rand(N, C, generator=torch.Generator().manual_seed(5), dtype=torch.float64))
        u = u * (gate.ref + a["gate_plus"]).repeat_interleave(HW, 0)
    y_ref = act_ref(u, act)
    if a["res"] is not None:
        res = k.inp(M, C, a["ldres"], a["res"], a["y_dtype"], k.rnd(M, C))
        y_ref = y_ref + res.ref
    y = k.out(M, C, a["ldy"], a["y"], a["y_dtype"])
    k.expect("y", y, y_ref)
    p = lambda o: None if o is None else o.ptr  # noqa: E731
    return lambda: lib.cabinet_affine_act(z.ptr, a["ldz"], a["z_dtype"], p(scale), p(shift), p(gate), a["gate_plus"], p(res),
                                          a["ldres"], y.ptr, a["ldy"], a["y_dtype"], M, HW, C, act, stream())


def run_add(lib, a, k):
    M, C, dt = a["M"], a["C"], a["dtype"]
    b = k.inp(M, C, a["ldb"], a["b"], dt, k.rnd(M, C))
    if a["inplace"]:   # out = a: the gradient fan-in adds into the region in place
        assert a["lda"] == a["ldo"] and a["a"] == a["out"]
        out = k.out(M, C, a["ldo"], a["out"], dt, acc=True)
        A = out
    else:
        A = k.inp(M, C, a["lda"], a["a"], dt, k.rnd(M, C))
        out = k.out(M, C, a["ldo"], a["out"], dt)
    k.expect("out", out, b.ref + (0 if a["inplace"] else A.ref))
    return lambda: lib.cabinet_add(A.ptr, a["lda"], b.ptr, a["ldb"], out.ptr, a["ldo"], dt, M, C, stream())


def run_col_sum(lib, a, k):
    M, C, dt = a["M"], a["C"], a["dtype"]
    x = k.inp(M, C, a["ldx"], a["x"], dt, k.rnd(M, C, shift=0.5))
    out = k.out(1, C, C, 0, F32, acc=a["accumulate"])
    sc = scratch(lib, M, C, 1)
    k.expect("out", out, x.ref.sum(0), red_tol(M))
    return lambda: lib.cabinet_col_sum(x.ptr, a["ldx"], dt, M, C, out.ptr, a["accumulate"], sc.data_ptr(), stream())


def _gate_inputs(a, k):
    N, HW, C, dt = a["N"], a["HW"], a["C"], a["dtype"]
    v = k.inp(N * HW, C, a["ldv"], a["v"], dt, k.rnd(N * HW, C, scale=2.0))
    dy = k.inp(N * HW, C, a["lddy"], a["dy"], dt, k.rnd(N * HW, C))
    s = k.inp(N, C, C, 0, F32, torch.rand(N, C, generator=torch.Generator().manual_seed(11), dtype=torch.float64))
    sp = (s.ref + a["plus"]).repeat_interleave(HW, 0)
    u = (v.ref * sp).requires_grad_(True)
    act_ref(u, a["act"]).backward(dy.ref)
    return N, HW, C, dt, v, dy, s, sp, u.grad


def run_gate_scale_backward(lib, a, k):
    N, HW, C, dt, v, dy, s, _, du = _gate_inputs(a, k)
    ds = k.out(N, C, C, 0, F32)
    k.expect("ds", ds, (du * v.ref).reshape(N, HW, C).sum(1), red_tol(HW))
    sc = torch.empty(N * int(lib.cabinet_train_scratch_floats(HW, C, 1)), device="cuda")
    return lambda: lib.cabinet_gate_scale_backward(dy.ptr, a["lddy"], v.ptr, a["ldv"], dt, s.ptr, a["plus"], a["act"],
                                                   ds.ptr, N, HW, C, sc.data_ptr(), stream())


def run_gate_apply_backward(lib, a, k):
    assert a["s"] is not None
    N, HW, C, dt, v, dy, s, sp, du = _gate_inputs(a, k)
    ref = du * sp
    dm = None
    if a["dm"] is not None:
        dm = k.inp(N, C, C, 0, F32, k.rnd(N, C))
        ref = ref + (dm.ref * a["inv_hw"]).repeat_interleave(HW, 0)
    dv = k.out(N * HW, C, a["lddv"], a["dv"], dt, acc=a["accumulate"])
    k.expect("dv", dv, ref)
    return lambda: lib.cabinet_gate_apply_backward(dy.ptr, a["lddy"], v.ptr, a["ldv"], dt, s.ptr, a["plus"],
                                                   None if dm is None else dm.ptr, a["inv_hw"], a["act"], dv.ptr,
                                                   a["lddv"], N, HW, C, a["accumulate"], stream())


def run_gate_mlp_backward(lib, a, k):
    N, C, J, gate = a["N"], a["C"], a["J"], a["gate"]
    HW = round(1.0 / a["mean_scale"])
    m = k.rnd(N, C).requires_grad_(True)
    w1, w2 = k.rnd(J, C, scale=0.4).requires_grad_(True), k.rnd(C, J, scale=0.6).requires_grad_(True)
    b1 = k.rnd(J, scale=0.3).requires_grad_(True) if a["db1"] is not None else None
    b2 = k.rnd(C, scale=0.3).requires_grad_(True) if a["db2"] is not None else None
    h = F.relu(F.linear(m, w1, b1))
    s = act_ref(F.linear(h, w2, b2), gate)
    ds_v = k.rnd(N, C)
    s.backward(ds_v)
    sums = k.vec(m.detach() * HW)
    w1d, w2d = k.vec(w1.detach()), k.vec(w2.detach())
    hd, sd, dsd = k.vec(h.detach()), k.vec(s.detach()), k.vec(ds_v)
    dw1, dw2 = k.out(J, C, C, 0, F32, acc=True), k.out(C, J, J, 0, F32, acc=True)
    db1 = k.out(1, J, J, 0, F32, acc=True) if b1 is not None else None
    db2 = k.out(1, C, C, 0, F32, acc=True) if b2 is not None else None
    dmean = k.out(N, C, C, 0, F32)
    for nm, op, t in (("dw1", dw1, w1), ("dw2", dw2, w2), ("db1", db1, b1), ("db2", db2, b2), ("dmean", dmean, m)):
        if op is not None:
            k.expect(nm, op, t.grad)
    sc = torch.empty(N * (C + J), device="cuda")
    p = lambda o: None if o is None else o.ptr  # noqa: E731
    return lambda: lib.cabinet_gate_mlp_backward(sums.ptr, a["mean_scale"], w1d.ptr, w2d.ptr, hd.ptr, sd.ptr, dsd.ptr, gate,
                                                 N, C, J, dw1.ptr, p(db1), dw2.ptr, p(db2), dmean.ptr, sc.data_ptr(),
                                                 stream())


def run_cab_combine_backward(lib, a, k):
    n, C, dt = a["n_pixels"], a["C"], a["dtype"]
    dout = k.inp(n, C, a["ldo"], a["dout"], dt, k.rnd(n, C))
    g, x, r = (k.inp(n, C, C, 0, dt, k.rnd(n, C, scale=2.0)) for _ in range(3))
    gamma = k.vec(torch.tensor([0.7]))
    dg, dr = k.out(n, C, C, 0, dt), k.out(n, C, C, 0, dt)
    dx = k.out(n, C, C, 0, dt, acc=a["accumulate_dx"])
    dgamma = k.out(1, 1, 1, 0, F32, acc=True)
    sig = torch.sigmoid(r.ref)
    k.expect("dg", dg, gamma.ref[0, 0] * dout.ref)
    k.expect("dx", dx, dout.ref * (1 + sig))
    k.expect("dr", dr, dout.ref * x.ref * sig * (1 - sig))
    k.expect("dgamma", dgamma, (dout.ref * g.ref).sum().reshape(1, 1), red_tol(n * C))
    sc = scratch(lib, n, C, 1)
    return lambda: lib.cabinet_cab_combine_backward(dout.ptr, a["ldo"], g.ptr, x.ptr, r.ptr, gamma.ptr, dt, dg.ptr, dx.ptr,
                                                    dr.ptr, dgamma.ptr, n, C, a["accumulate_dx"], sc.data_ptr(), stream())


def run_softmax_backward(lib, a, k):
    rows, cols, alpha = a["rows"], a["cols"], a["alpha"]
    p = k.inp(rows, cols, cols, 0, F32, torch.softmax(k.rnd(rows, cols, scale=3.0), -1))
    dp = k.inp(rows, cols, cols, 0, F32, k.rnd(rows, cols))
    ds = k.out(rows, cols, cols, 0, F32)
    k.expect("ds", ds, p.ref * (dp.ref - (dp.ref * p.ref).sum(-1, keepdim=True)) * alpha)
    return lambda: lib.cabinet_softmax_backward(p.ptr, dp.ptr, ds.ptr, rows, cols, alpha, stream())


def run_conv_dgrad(lib, a, k):
    N, H, W, Cin, Cout, KH, KW = (a[n] for n in ("N", "H", "W", "Cin", "Cout", "KH", "KW"))
    s, pad, OH, OW, dt = a["stride"], a["pad"], a["OH"], a["OW"], a["dtype"]
    assert a["w_sco"] == KH * KW * a["w_stap"] and a["w_stap"] >= Cin
    w = k.rnd(Cout, Cin, KH, KW, scale=(Cin * KH * KW) ** -0.5).to(TD[a["w_dtype"]]).double()
    packed = torch.zeros(Cout, KH * KW, a["w_stap"], dtype=torch.float64)
    packed[:, :, :Cin] = w.permute(0, 2, 3, 1).reshape(Cout, KH * KW, Cin)
    wp = k.inp(1, packed.numel(), packed.numel(), a["w_packed"], a["w_dtype"], packed.reshape(1, -1))
    dy = k.inp(N * OH * OW, Cout, a["lddy"], a["dy"], dt, k.rnd(N * OH * OW, Cout))
    dx = k.out(N * H * W, Cin, a["lddx"], a["dx"], dt, acc=a["accumulate"])
    ref = torch.nn.grad.conv2d_input((N, Cin, H, W), w, nchw(dy.ref, N, OH, OW), s, pad)
    k.expect("dx", dx, rows_of(ref))
    return lambda: lib.cabinet_conv_dgrad(dy.ptr, a["lddy"], dt, wp.ptr, a["w_dtype"], a["w_sco"], a["w_stap"], dx.ptr,
                                          a["lddx"], N, H, W, Cin, Cout, KH, KW, s, pad, OH, OW, a["accumulate"], stream())


def run_conv_wgrad(lib, a, k):
    N, H, W, Cin, Cout, KH, KW = (a[n] for n in ("N", "H", "W", "Cin", "Cout", "KH", "KW"))
    s, pad, OH, OW, dt, xdt = a["stride"], a["pad"], a["OH"], a["OW"], a["dtype"], a["x_dtype"]
    dy = k.inp(N * OH * OW, Cout, a["lddy"], a["dy"], dt, k.rnd(N * OH * OW, Cout))
    if a["sxc"] == 1:   # NHWC map, pixel stride sxw
        assert a["sxh"] == W * a["sxw"] and a["sxn"] == H * a["sxh"]
        x = k.inp(N * H * W, Cin, a["sxw"], a["x"], xdt, k.rnd(N * H * W, Cin))
        x4 = nchw(x.ref, N, H, W)
    else:               # the dense fp32 NCHW network input
        assert (a["sxn"], a["sxh"], a["sxw"], a["sxc"]) == (Cin * H * W, W, 1, H * W)
        x = k.inp(1, N * Cin * H * W, N * Cin * H * W, a["x"], xdt, k.rnd(1, N * Cin * H * W))
        x4 = x.ref.reshape(N, Cin, H, W)
    dw = k.out(Cout, Cin * KH * KW, Cin * KH * KW, 0, F32, acc=True)
    ref = torch.nn.grad.conv2d_weight(x4, (Cout, Cin, KH, KW), nchw(dy.ref, N, OH, OW), s, pad)
    k.expect("dw", dw, ref.reshape(Cout, -1), red_tol(N * OH * OW))
    sc = torch.empty(int(lib.cabinet_conv_wgrad_scratch_floats(N, OH, OW, Cin, Cout, KH, KW)), device="cuda")
    return lambda: lib.cabinet_conv_wgrad(dy.ptr, a["lddy"], dt, x.ptr, xdt, a["sxn"], a["sxh"], a["sxw"], a["sxc"], dw.ptr,
                                          N, H, W, Cin, Cout, KH, KW, s, pad, OH, OW, sc.data_ptr(), stream())


def run_dwconv_dgrad(lib, a, k):
    N, H, W, C, kk, s, OH, OW, dt = (a[n] for n in ("N", "H", "W", "C", "k", "stride", "OH", "OW", "dtype"))
    w = k.rnd(C, 1, kk, kk, scale=1.0 / kk).float().double()
    wp = k.inp(kk * kk, C, C, a["w_packed"], F32, w.reshape(C, kk * kk).t())
    dy = k.inp(N * OH * OW, C, a["lddy"], a["dy"], dt, k.rnd(N * OH * OW, C))
    dx = k.out(N * H * W, C, a["lddx"], a["dx"], dt, acc=a["accumulate"])
    ref = torch.nn.grad.conv2d_input((N, C, H, W), w, nchw(dy.ref, N, OH, OW), s, (kk - 1) // 2, groups=C)
    k.expect("dx", dx, rows_of(ref))
    return lambda: lib.cabinet_dwconv_dgrad(dy.ptr, a["lddy"], dt, wp.ptr, dx.ptr, a["lddx"], N, H, W, C, kk, s, OH, OW,
                                            a["accumulate"], stream())


def run_dwconv_wgrad(lib, a, k):
    N, H, W, C, kk, s, OH, OW, dt = (a[n] for n in ("N", "H", "W", "C", "k", "stride", "OH", "OW", "dtype"))
    dy = k.inp(N * OH * OW, C, a["lddy"], a["dy"], dt, k.rnd(N * OH * OW, C))
    x = k.inp(N * H * W, C, a["ldx"], a["x"], dt, k.rnd(N * H * W, C))
    dw = k.out(C, kk * kk, kk * kk, 0, F32, acc=True)
    ref = torch.nn.grad.conv2d_weight(nchw(x.ref, N, H, W), (C, 1, kk, kk), nchw(dy.ref, N, OH, OW), s, (kk - 1) // 2,
                                      groups=C)
    k.expect("dw", dw, ref.reshape(C, -1), red_tol(N * OH * OW))
    sc = scratch(lib, N * OH * OW, C, kk * kk)
    return lambda: lib.cabinet_dwconv_wgrad(dy.ptr, a["lddy"], x.ptr, a["ldx"], dt, dw.ptr, N, H, W, C, kk, s, OH, OW,
                                            sc.data_ptr(), stream())


def _operator(op):
    kind, n_in, n_out, transpose = op
    m = np.eye(n_in) if kind == "identity" else (bilinear_matrix if kind == "bilinear" else adaptive_pool_matrix)(n_in, n_out)
    m = torch.from_numpy(m.T if transpose else m).float().double()   # the tables hold fp32 weights
    nz = [torch.nonzero(r).flatten() for r in m]
    tabs = (np.cumsum([0] + [len(i) for i in nz]).astype(np.int32), torch.cat(nz).numpy().astype(np.int32),
            torch.cat([r[i] for r, i in zip(m, nz)]).float().numpy())
    return m, [torch.from_numpy(t).cuda() for t in tabs]


def run_resample_sep(lib, a, k):
    N, OH, OW, C, flags = a["N"], a["OH"], a["OW"], a["C"], a["accumulate"]
    (my, (ys, yi, yw)), (mx, (xs, xi, xw)) = _operator(a["y_op"]), _operator(a["x_op"])
    assert my.shape[0] == OH and mx.shape[0] == OW and a["osc"] == 1
    IH, IW = my.shape[1], mx.shape[1]
    if a["isc"] == 1:   # NHWC map, pixel stride isx
        assert a["isy"] == IW * a["isx"] and a["isn"] == IH * a["isy"]
        x = k.inp(N * IH * IW, C, a["isx"], a["in"], a["in_dtype"], k.rnd(N * IH * IW, C))
        x4 = x.ref.reshape(N, IH, IW, C)
    else:               # planar [N][C][IH][IW]
        assert (a["isn"], a["isy"], a["isx"], a["isc"]) == (C * IH * IW, IW, 1, IH * IW)
        x = k.inp(1, N * C * IH * IW, N * C * IH * IW, a["in"], a["in_dtype"], k.rnd(1, N * C * IH * IW))
        x4 = x.ref.reshape(N, C, IH, IW).permute(0, 2, 3, 1)
    assert a["osy"] == OW * a["osx"] and a["osn"] == OH * a["osy"]
    out = k.out(N * OH * OW, C, a["osx"], a["out"], a["out_dtype"], acc=flags & 1)
    k.expect("out", out, torch.einsum("ai,bj,nijc->nabc", my, mx, x4).reshape(-1, C))
    return lambda: lib.cabinet_resample_sep(x.ptr, a["in_dtype"], a["isn"], a["isy"], a["isx"], a["isc"], out.ptr,
                                            a["out_dtype"], a["osn"], a["osy"], a["osx"], a["osc"], N, OH, OW, C,
                                            ys.data_ptr(), yi.data_ptr(), yw.data_ptr(), xs.data_ptr(), xi.data_ptr(),
                                            xw.data_ptr(), flags, stream())


def run_channel_sum(lib, a, k):
    N, HW, C, dt = a["N"], a["HW"], a["C"], a["dtype"]
    x = k.inp(N * HW, C, a["ldx"], a["x"], dt, k.rnd(N * HW, C, shift=0.5))
    out = k.out(N, C, C, 0, F32)
    k.expect("out", out, x.ref.reshape(N, HW, C).sum(1), red_tol(HW))
    nbytes = 256 + N * 64 * C * 4 + 4096
    sc = torch.zeros(nbytes // 4, device="cuda")
    return lambda: lib.cabinet_channel_sum(x.ptr, a["ldx"], dt, N, HW, C, out.ptr, sc.data_ptr(), nbytes, stream())


RUNNERS = {name[4:]: fn for name, fn in globals().items() if name.startswith("run_")}


# One case per variant key: the smallest recorded call of each (tests/test_train_variants_cpu.py lists any key
# the step reaches that is missing here, with an example call).
CASES = [
    ('bn_train_stats', {'x': 0, 'ldx': 96, 'dtype': 1, 'M': 12, 'C': 96, 'gamma': 0, 'beta': 0, 'eps': 1e-05,
                        'momentum': 0.1, 'running_mean': 0, 'running_var': 0, 'stats': 0}),
    ('bn_train_stats', {'x': 0, 'ldx': 64, 'dtype': 1, 'M': 16384, 'C': 64, 'gamma': 0, 'beta': 0, 'eps': 1e-05,
                        'momentum': 0.1, 'running_mean': 0, 'running_var': 0, 'stats': 0}),
    ('bn_train_stats', {'x': 0, 'ldx': 96, 'dtype': 2, 'M': 12, 'C': 96, 'gamma': 0, 'beta': 0, 'eps': 1e-05,
                        'momentum': 0.1, 'running_mean': 0, 'running_var': 0, 'stats': 0}),
    ('bn_train_stats', {'x': 0, 'ldx': 64, 'dtype': 2, 'M': 16384, 'C': 64, 'gamma': 0, 'beta': 0, 'eps': 1e-05,
                        'momentum': 0.1, 'running_mean': 0, 'running_var': 0, 'stats': 0}),
    ('bn_train_stats', {'x': 0, 'ldx': 96, 'dtype': 0, 'M': 12, 'C': 96, 'gamma': 0, 'beta': 0, 'eps': 1e-05,
                        'momentum': 0.1, 'running_mean': 0, 'running_var': 0, 'stats': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 96, 'z': 0, 'ldz': 96, 'dtype': 1, 'stats': 0, 'act': 0, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 96, 'M': 12, 'C': 96, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 128, 'z': 0, 'ldz': 128, 'dtype': 1, 'stats': 0, 'act': 1, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 128, 'M': 12, 'C': 128, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 120, 'z': 0, 'ldz': 120, 'dtype': 1, 'stats': 0, 'act': 2, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 120, 'M': 48, 'C': 120, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 16, 'z': 0, 'ldz': 16, 'dtype': 1, 'stats': 0, 'act': 0, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 16, 'M': 65536, 'C': 16, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 256, 'z': 0, 'ldz': 256, 'dtype': 1, 'stats': 0, 'act': 1, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 256, 'M': 4096, 'C': 256, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 16, 'z': 0, 'ldz': 16, 'dtype': 1, 'stats': 0, 'act': 2, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 16, 'M': 65536, 'C': 16, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 384, 'z': 0, 'ldz': 128, 'dtype': 1, 'stats': 0, 'act': 1, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 128, 'M': 192, 'C': 128, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 832, 'z': 0, 'ldz': 576, 'dtype': 1, 'stats': 0, 'act': 2, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 576, 'M': 12, 'C': 576, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 96, 'z': 0, 'ldz': 96, 'dtype': 2, 'stats': 0, 'act': 0, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 96, 'M': 12, 'C': 96, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 128, 'z': 0, 'ldz': 128, 'dtype': 2, 'stats': 0, 'act': 1, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 128, 'M': 12, 'C': 128, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 120, 'z': 0, 'ldz': 120, 'dtype': 2, 'stats': 0, 'act': 2, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 120, 'M': 48, 'C': 120, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 16, 'z': 0, 'ldz': 16, 'dtype': 2, 'stats': 0, 'act': 0, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 16, 'M': 65536, 'C': 16, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 256, 'z': 0, 'ldz': 256, 'dtype': 2, 'stats': 0, 'act': 1, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 256, 'M': 4096, 'C': 256, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 16, 'z': 0, 'ldz': 16, 'dtype': 2, 'stats': 0, 'act': 2, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 16, 'M': 65536, 'C': 16, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 384, 'z': 0, 'ldz': 128, 'dtype': 2, 'stats': 0, 'act': 1, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 128, 'M': 192, 'C': 128, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 832, 'z': 0, 'ldz': 576, 'dtype': 2, 'stats': 0, 'act': 2, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 576, 'M': 12, 'C': 576, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 96, 'z': 0, 'ldz': 96, 'dtype': 0, 'stats': 0, 'act': 0, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 96, 'M': 12, 'C': 96, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 128, 'z': 0, 'ldz': 128, 'dtype': 0, 'stats': 0, 'act': 1, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 128, 'M': 12, 'C': 128, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 120, 'z': 0, 'ldz': 120, 'dtype': 0, 'stats': 0, 'act': 2, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 120, 'M': 48, 'C': 120, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 384, 'z': 0, 'ldz': 128, 'dtype': 0, 'stats': 0, 'act': 1, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 128, 'M': 192, 'C': 128, 'accumulate': 0}),
    ('bn_train_backward', {'dy': 0, 'lddy': 832, 'z': 0, 'ldz': 576, 'dtype': 0, 'stats': 0, 'act': 2, 'dgamma': 0,
                           'dbeta': 0, 'dz': 0, 'lddz': 576, 'M': 12, 'C': 576, 'accumulate': 0}),
    ('bn_frozen_backward', {'dy': 0, 'lddy': 160, 'z': 0, 'ldz': 160, 'dtype': 1, 'stats': 0, 'act': 0, 'dgamma': 0,
                            'dbeta': 0, 'dz': 0, 'lddz': 160, 'M': 256, 'C': 160, 'accumulate': 0}),
    ('bn_frozen_backward', {'dy': 0, 'lddy': 128, 'z': 0, 'ldz': 128, 'dtype': 1, 'stats': 0, 'act': 1, 'dgamma': 0,
                            'dbeta': 0, 'dz': 0, 'lddz': 128, 'M': 256, 'C': 128, 'accumulate': 0}),
    ('bn_frozen_backward', {'dy': 0, 'lddy': 184, 'z': 0, 'ldz': 184, 'dtype': 1, 'stats': 0, 'act': 2, 'dgamma': 0,
                            'dbeta': 0, 'dz': 0, 'lddz': 184, 'M': 1024, 'C': 184, 'accumulate': 0}),
    ('bn_frozen_backward', {'dy': 0, 'lddy': 384, 'z': 0, 'ldz': 128, 'dtype': 1, 'stats': 0, 'act': 1, 'dgamma': 0,
                            'dbeta': 0, 'dz': 0, 'lddz': 128, 'M': 4096, 'C': 128, 'accumulate': 0}),
    ('bn_frozen_backward', {'dy': 0, 'lddy': 1216, 'z': 0, 'ldz': 960, 'dtype': 1, 'stats': 0, 'act': 2, 'dgamma': 0,
                            'dbeta': 0, 'dz': 0, 'lddz': 960, 'M': 256, 'C': 960, 'accumulate': 0}),
    ('bn_frozen_backward', {'dy': 0, 'lddy': 160, 'z': 0, 'ldz': 160, 'dtype': 0, 'stats': 0, 'act': 0, 'dgamma': 0,
                            'dbeta': 0, 'dz': 0, 'lddz': 160, 'M': 256, 'C': 160, 'accumulate': 0}),
    ('bn_frozen_backward', {'dy': 0, 'lddy': 128, 'z': 0, 'ldz': 128, 'dtype': 0, 'stats': 0, 'act': 1, 'dgamma': 0,
                            'dbeta': 0, 'dz': 0, 'lddz': 128, 'M': 256, 'C': 128, 'accumulate': 0}),
    ('bn_frozen_backward', {'dy': 0, 'lddy': 184, 'z': 0, 'ldz': 184, 'dtype': 0, 'stats': 0, 'act': 2, 'dgamma': 0,
                            'dbeta': 0, 'dz': 0, 'lddz': 184, 'M': 1024, 'C': 184, 'accumulate': 0}),
    ('bn_frozen_backward', {'dy': 0, 'lddy': 384, 'z': 0, 'ldz': 128, 'dtype': 0, 'stats': 0, 'act': 1, 'dgamma': 0,
                            'dbeta': 0, 'dz': 0, 'lddz': 128, 'M': 4096, 'C': 128, 'accumulate': 0}),
    ('bn_frozen_backward', {'dy': 0, 'lddy': 1216, 'z': 0, 'ldz': 960, 'dtype': 0, 'stats': 0, 'act': 2, 'dgamma': 0,
                            'dbeta': 0, 'dz': 0, 'lddz': 960, 'M': 256, 'C': 960, 'accumulate': 0}),
    ('affine_act', {'z': 0, 'ldz': 96, 'z_dtype': 1, 'scale': 0, 'shift': 0, 'gate': None, 'gate_plus': 0.0, 'res': 0,
                    'ldres': 96, 'y': 0, 'ldy': 96, 'y_dtype': 1, 'M': 12, 'HW': 6, 'C': 96, 'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 96, 'z_dtype': 1, 'scale': 0, 'shift': 0, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 96, 'y_dtype': 1, 'M': 12, 'HW': 6, 'C': 96, 'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 128, 'z_dtype': 1, 'scale': 0, 'shift': 0, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 128, 'y_dtype': 1, 'M': 12, 'HW': 6, 'C': 128, 'act': 1}),
    ('affine_act', {'z': 0, 'ldz': 120, 'z_dtype': 1, 'scale': 0, 'shift': 0, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 120, 'y_dtype': 1, 'M': 48, 'HW': 24, 'C': 120, 'act': 2}),
    ('affine_act', {'z': 0, 'ldz': 16, 'z_dtype': 1, 'scale': None, 'shift': None, 'gate': 0, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 16, 'y_dtype': 1, 'M': 768, 'HW': 384, 'C': 16, 'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 72, 'z_dtype': 1, 'scale': None, 'shift': None, 'gate': 0, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 72, 'y_dtype': 1, 'M': 4096, 'HW': 2048, 'C': 72,
                    'act': 1}),
    ('affine_act', {'z': 0, 'ldz': 288, 'z_dtype': 1, 'scale': None, 'shift': None, 'gate': 0, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 288, 'y_dtype': 1, 'M': 12, 'HW': 6, 'C': 288, 'act': 2}),
    ('affine_act', {'z': 0, 'ldz': 256, 'z_dtype': 1, 'scale': None, 'shift': None, 'gate': 0, 'gate_plus': 1.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 256, 'y_dtype': 1, 'M': 192, 'HW': 96, 'C': 256,
                    'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 96, 'z_dtype': 1, 'scale': None, 'shift': None, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 96, 'y_dtype': 1, 'M': 12, 'HW': 6, 'C': 96, 'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 128, 'z_dtype': 1, 'scale': 0, 'shift': 0, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 384, 'y_dtype': 1, 'M': 192, 'HW': 96, 'C': 128,
                    'act': 1}),
    ('affine_act', {'z': 0, 'ldz': 576, 'z_dtype': 1, 'scale': 0, 'shift': 0, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 832, 'y_dtype': 1, 'M': 12, 'HW': 6, 'C': 576, 'act': 2}),
    ('affine_act', {'z': 0, 'ldz': 128, 'z_dtype': 1, 'scale': None, 'shift': None, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 640, 'y_dtype': 1, 'M': 12, 'HW': 6, 'C': 128, 'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 96, 'z_dtype': 2, 'scale': 0, 'shift': 0, 'gate': None, 'gate_plus': 0.0, 'res': 0,
                    'ldres': 96, 'y': 0, 'ldy': 96, 'y_dtype': 2, 'M': 12, 'HW': 6, 'C': 96, 'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 96, 'z_dtype': 2, 'scale': 0, 'shift': 0, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 96, 'y_dtype': 2, 'M': 12, 'HW': 6, 'C': 96, 'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 128, 'z_dtype': 2, 'scale': 0, 'shift': 0, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 128, 'y_dtype': 2, 'M': 12, 'HW': 6, 'C': 128, 'act': 1}),
    ('affine_act', {'z': 0, 'ldz': 120, 'z_dtype': 2, 'scale': 0, 'shift': 0, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 120, 'y_dtype': 2, 'M': 48, 'HW': 24, 'C': 120, 'act': 2}),
    ('affine_act', {'z': 0, 'ldz': 16, 'z_dtype': 2, 'scale': None, 'shift': None, 'gate': 0, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 16, 'y_dtype': 2, 'M': 768, 'HW': 384, 'C': 16, 'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 72, 'z_dtype': 2, 'scale': None, 'shift': None, 'gate': 0, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 72, 'y_dtype': 2, 'M': 4096, 'HW': 2048, 'C': 72,
                    'act': 1}),
    ('affine_act', {'z': 0, 'ldz': 288, 'z_dtype': 2, 'scale': None, 'shift': None, 'gate': 0, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 288, 'y_dtype': 2, 'M': 12, 'HW': 6, 'C': 288, 'act': 2}),
    ('affine_act', {'z': 0, 'ldz': 256, 'z_dtype': 2, 'scale': None, 'shift': None, 'gate': 0, 'gate_plus': 1.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 256, 'y_dtype': 2, 'M': 192, 'HW': 96, 'C': 256,
                    'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 96, 'z_dtype': 2, 'scale': None, 'shift': None, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 96, 'y_dtype': 2, 'M': 12, 'HW': 6, 'C': 96, 'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 128, 'z_dtype': 2, 'scale': 0, 'shift': 0, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 384, 'y_dtype': 2, 'M': 192, 'HW': 96, 'C': 128,
                    'act': 1}),
    ('affine_act', {'z': 0, 'ldz': 576, 'z_dtype': 2, 'scale': 0, 'shift': 0, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 832, 'y_dtype': 2, 'M': 12, 'HW': 6, 'C': 576, 'act': 2}),
    ('affine_act', {'z': 0, 'ldz': 128, 'z_dtype': 2, 'scale': None, 'shift': None, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 640, 'y_dtype': 2, 'M': 12, 'HW': 6, 'C': 128, 'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 8, 'z_dtype': 0, 'scale': None, 'shift': None, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 8, 'y_dtype': 1, 'M': 12, 'HW': 6, 'C': 8, 'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 5, 'z_dtype': 0, 'scale': None, 'shift': None, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 8, 'y_dtype': 1, 'M': 256, 'HW': 128, 'C': 5, 'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 8, 'z_dtype': 0, 'scale': None, 'shift': None, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 8, 'y_dtype': 2, 'M': 12, 'HW': 6, 'C': 8, 'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 5, 'z_dtype': 0, 'scale': None, 'shift': None, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 8, 'y_dtype': 2, 'M': 256, 'HW': 128, 'C': 5, 'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 96, 'z_dtype': 0, 'scale': 0, 'shift': 0, 'gate': None, 'gate_plus': 0.0, 'res': 0,
                    'ldres': 96, 'y': 0, 'ldy': 96, 'y_dtype': 0, 'M': 12, 'HW': 6, 'C': 96, 'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 96, 'z_dtype': 0, 'scale': 0, 'shift': 0, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 96, 'y_dtype': 0, 'M': 12, 'HW': 6, 'C': 96, 'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 128, 'z_dtype': 0, 'scale': 0, 'shift': 0, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 128, 'y_dtype': 0, 'M': 12, 'HW': 6, 'C': 128, 'act': 1}),
    ('affine_act', {'z': 0, 'ldz': 120, 'z_dtype': 0, 'scale': 0, 'shift': 0, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 120, 'y_dtype': 0, 'M': 48, 'HW': 24, 'C': 120, 'act': 2}),
    ('affine_act', {'z': 0, 'ldz': 16, 'z_dtype': 0, 'scale': None, 'shift': None, 'gate': 0, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 16, 'y_dtype': 0, 'M': 768, 'HW': 384, 'C': 16, 'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 72, 'z_dtype': 0, 'scale': None, 'shift': None, 'gate': 0, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 72, 'y_dtype': 0, 'M': 4096, 'HW': 2048, 'C': 72,
                    'act': 1}),
    ('affine_act', {'z': 0, 'ldz': 288, 'z_dtype': 0, 'scale': None, 'shift': None, 'gate': 0, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 288, 'y_dtype': 0, 'M': 12, 'HW': 6, 'C': 288, 'act': 2}),
    ('affine_act', {'z': 0, 'ldz': 256, 'z_dtype': 0, 'scale': None, 'shift': None, 'gate': 0, 'gate_plus': 1.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 256, 'y_dtype': 0, 'M': 192, 'HW': 96, 'C': 256,
                    'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 96, 'z_dtype': 0, 'scale': None, 'shift': None, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 96, 'y_dtype': 0, 'M': 12, 'HW': 6, 'C': 96, 'act': 0}),
    ('affine_act', {'z': 0, 'ldz': 128, 'z_dtype': 0, 'scale': 0, 'shift': 0, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 384, 'y_dtype': 0, 'M': 192, 'HW': 96, 'C': 128,
                    'act': 1}),
    ('affine_act', {'z': 0, 'ldz': 576, 'z_dtype': 0, 'scale': 0, 'shift': 0, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 832, 'y_dtype': 0, 'M': 12, 'HW': 6, 'C': 576, 'act': 2}),
    ('affine_act', {'z': 0, 'ldz': 128, 'z_dtype': 0, 'scale': None, 'shift': None, 'gate': None, 'gate_plus': 0.0,
                    'res': None, 'ldres': 0, 'y': 0, 'ldy': 640, 'y_dtype': 0, 'M': 12, 'HW': 6, 'C': 128, 'act': 0}),
    ('add', {'a': 0, 'lda': 256, 'b': 0, 'ldb': 256, 'out': 0, 'ldo': 256, 'dtype': 1, 'M': 12, 'C': 256,
             'inplace': True}),
    ('add', {'a': 0, 'lda': 128, 'b': 0, 'ldb': 640, 'out': 0, 'ldo': 128, 'dtype': 1, 'M': 12, 'C': 128,
             'inplace': True}),
    ('add', {'a': 0, 'lda': 256, 'b': 0, 'ldb': 256, 'out': 0, 'ldo': 256, 'dtype': 2, 'M': 12, 'C': 256,
             'inplace': True}),
    ('add', {'a': 0, 'lda': 128, 'b': 0, 'ldb': 640, 'out': 0, 'ldo': 128, 'dtype': 2, 'M': 12, 'C': 128,
             'inplace': True}),
    ('add', {'a': 0, 'lda': 128, 'b': 0, 'ldb': 640, 'out': 0, 'ldo': 128, 'dtype': 0, 'M': 12, 'C': 128,
             'inplace': True}),
    ('col_sum', {'x': 0, 'ldx': 256, 'dtype': 1, 'M': 12, 'C': 256, 'out': 0, 'accumulate': 1}),
    ('col_sum', {'x': 0, 'ldx': 256, 'dtype': 2, 'M': 12, 'C': 256, 'out': 0, 'accumulate': 1}),
    ('col_sum', {'x': 0, 'ldx': 8, 'dtype': 0, 'M': 12, 'C': 8, 'out': 0, 'accumulate': 1}),
    ('col_sum', {'x': 0, 'ldx': 5, 'dtype': 0, 'M': 256, 'C': 5, 'out': 0, 'accumulate': 1}),
    ('gate_scale_backward', {'dy': 0, 'lddy': 16, 'v': 0, 'ldv': 16, 'dtype': 1, 's': 0, 'plus': 0.0, 'act': 0,
                             'ds': 0, 'N': 2, 'HW': 384, 'C': 16}),
    ('gate_scale_backward', {'dy': 0, 'lddy': 256, 'v': 0, 'ldv': 256, 'dtype': 1, 's': 0, 'plus': 1.0, 'act': 0,
                             'ds': 0, 'N': 2, 'HW': 96, 'C': 256}),
    ('gate_scale_backward', {'dy': 0, 'lddy': 72, 'v': 0, 'ldv': 72, 'dtype': 1, 's': 0, 'plus': 0.0, 'act': 1,
                             'ds': 0, 'N': 2, 'HW': 2048, 'C': 72}),
    ('gate_scale_backward', {'dy': 0, 'lddy': 288, 'v': 0, 'ldv': 288, 'dtype': 1, 's': 0, 'plus': 0.0, 'act': 2,
                             'ds': 0, 'N': 2, 'HW': 6, 'C': 288}),
    ('gate_scale_backward', {'dy': 0, 'lddy': 16, 'v': 0, 'ldv': 16, 'dtype': 2, 's': 0, 'plus': 0.0, 'act': 0,
                             'ds': 0, 'N': 2, 'HW': 384, 'C': 16}),
    ('gate_scale_backward', {'dy': 0, 'lddy': 256, 'v': 0, 'ldv': 256, 'dtype': 2, 's': 0, 'plus': 1.0, 'act': 0,
                             'ds': 0, 'N': 2, 'HW': 96, 'C': 256}),
    ('gate_scale_backward', {'dy': 0, 'lddy': 72, 'v': 0, 'ldv': 72, 'dtype': 2, 's': 0, 'plus': 0.0, 'act': 1,
                             'ds': 0, 'N': 2, 'HW': 2048, 'C': 72}),
    ('gate_scale_backward', {'dy': 0, 'lddy': 288, 'v': 0, 'ldv': 288, 'dtype': 2, 's': 0, 'plus': 0.0, 'act': 2,
                             'ds': 0, 'N': 2, 'HW': 6, 'C': 288}),
    ('gate_scale_backward', {'dy': 0, 'lddy': 16, 'v': 0, 'ldv': 16, 'dtype': 0, 's': 0, 'plus': 0.0, 'act': 0,
                             'ds': 0, 'N': 2, 'HW': 384, 'C': 16}),
    ('gate_scale_backward', {'dy': 0, 'lddy': 256, 'v': 0, 'ldv': 256, 'dtype': 0, 's': 0, 'plus': 1.0, 'act': 0,
                             'ds': 0, 'N': 2, 'HW': 96, 'C': 256}),
    ('gate_scale_backward', {'dy': 0, 'lddy': 72, 'v': 0, 'ldv': 72, 'dtype': 0, 's': 0, 'plus': 0.0, 'act': 1,
                             'ds': 0, 'N': 2, 'HW': 2048, 'C': 72}),
    ('gate_scale_backward', {'dy': 0, 'lddy': 288, 'v': 0, 'ldv': 288, 'dtype': 0, 's': 0, 'plus': 0.0, 'act': 2,
                             'ds': 0, 'N': 2, 'HW': 6, 'C': 288}),
    ('gate_apply_backward', {'dy': 0, 'lddy': 16, 'v': 0, 'ldv': 16, 'dtype': 1, 's': 0, 'plus': 0.0, 'dm': 0,
                             'inv_hw': 0.0026041666666666665, 'act': 0, 'dv': 0, 'lddv': 16, 'N': 2, 'HW': 384,
                             'C': 16, 'accumulate': 0}),
    ('gate_apply_backward', {'dy': 0, 'lddy': 72, 'v': 0, 'ldv': 72, 'dtype': 1, 's': 0, 'plus': 0.0, 'dm': 0,
                             'inv_hw': 0.00048828125, 'act': 1, 'dv': 0, 'lddv': 72, 'N': 2, 'HW': 2048, 'C': 72,
                             'accumulate': 0}),
    ('gate_apply_backward', {'dy': 0, 'lddy': 288, 'v': 0, 'ldv': 288, 'dtype': 1, 's': 0, 'plus': 0.0, 'dm': 0,
                             'inv_hw': 0.16666666666666666, 'act': 2, 'dv': 0, 'lddv': 288, 'N': 2, 'HW': 6, 'C': 288,
                             'accumulate': 0}),
    ('gate_apply_backward', {'dy': 0, 'lddy': 256, 'v': 0, 'ldv': 256, 'dtype': 1, 's': 0, 'plus': 1.0, 'dm': 0,
                             'inv_hw': 0.010416666666666666, 'act': 0, 'dv': 0, 'lddv': 256, 'N': 2, 'HW': 96,
                             'C': 256, 'accumulate': 0}),
    ('gate_apply_backward', {'dy': 0, 'lddy': 16, 'v': 0, 'ldv': 16, 'dtype': 2, 's': 0, 'plus': 0.0, 'dm': 0,
                             'inv_hw': 0.0026041666666666665, 'act': 0, 'dv': 0, 'lddv': 16, 'N': 2, 'HW': 384,
                             'C': 16, 'accumulate': 0}),
    ('gate_apply_backward', {'dy': 0, 'lddy': 72, 'v': 0, 'ldv': 72, 'dtype': 2, 's': 0, 'plus': 0.0, 'dm': 0,
                             'inv_hw': 0.00048828125, 'act': 1, 'dv': 0, 'lddv': 72, 'N': 2, 'HW': 2048, 'C': 72,
                             'accumulate': 0}),
    ('gate_apply_backward', {'dy': 0, 'lddy': 288, 'v': 0, 'ldv': 288, 'dtype': 2, 's': 0, 'plus': 0.0, 'dm': 0,
                             'inv_hw': 0.16666666666666666, 'act': 2, 'dv': 0, 'lddv': 288, 'N': 2, 'HW': 6, 'C': 288,
                             'accumulate': 0}),
    ('gate_apply_backward', {'dy': 0, 'lddy': 256, 'v': 0, 'ldv': 256, 'dtype': 2, 's': 0, 'plus': 1.0, 'dm': 0,
                             'inv_hw': 0.010416666666666666, 'act': 0, 'dv': 0, 'lddv': 256, 'N': 2, 'HW': 96,
                             'C': 256, 'accumulate': 0}),
    ('gate_apply_backward', {'dy': 0, 'lddy': 16, 'v': 0, 'ldv': 16, 'dtype': 0, 's': 0, 'plus': 0.0, 'dm': 0,
                             'inv_hw': 0.0026041666666666665, 'act': 0, 'dv': 0, 'lddv': 16, 'N': 2, 'HW': 384,
                             'C': 16, 'accumulate': 0}),
    ('gate_apply_backward', {'dy': 0, 'lddy': 72, 'v': 0, 'ldv': 72, 'dtype': 0, 's': 0, 'plus': 0.0, 'dm': 0,
                             'inv_hw': 0.00048828125, 'act': 1, 'dv': 0, 'lddv': 72, 'N': 2, 'HW': 2048, 'C': 72,
                             'accumulate': 0}),
    ('gate_apply_backward', {'dy': 0, 'lddy': 288, 'v': 0, 'ldv': 288, 'dtype': 0, 's': 0, 'plus': 0.0, 'dm': 0,
                             'inv_hw': 0.16666666666666666, 'act': 2, 'dv': 0, 'lddv': 288, 'N': 2, 'HW': 6, 'C': 288,
                             'accumulate': 0}),
    ('gate_apply_backward', {'dy': 0, 'lddy': 256, 'v': 0, 'ldv': 256, 'dtype': 0, 's': 0, 'plus': 1.0, 'dm': 0,
                             'inv_hw': 0.010416666666666666, 'act': 0, 'dv': 0, 'lddv': 256, 'N': 2, 'HW': 96,
                             'C': 256, 'accumulate': 0}),
    ('gate_mlp_backward', {'mean': 0, 'mean_scale': 0.0026041666666666665, 'w1': 0, 'w2': 0, 'hidden': 0, 's': 0,
                           'ds': 0, 'gate': 3, 'N': 2, 'C': 16, 'J': 8, 'dw1': 0, 'db1': 0, 'dw2': 0, 'db2': 0,
                           'dmean': 0}),
    ('gate_mlp_backward', {'mean': 0, 'mean_scale': 0.00048828125, 'w1': 0, 'w2': 0, 'hidden': 0, 's': 0, 'ds': 0,
                           'gate': 4, 'N': 2, 'C': 256, 'J': 64, 'dw1': 0, 'db1': None, 'dw2': 0, 'db2': None,
                           'dmean': 0}),
    ('cab_combine_backward', {'dout': 0, 'ldo': 832, 'g': 0, 'x': 0, 'r': 0, 'gamma': 0, 'dtype': 1, 'dg': 0, 'dx': 0,
                              'dr': 0, 'dgamma': 0, 'n_pixels': 12, 'C': 256, 'accumulate_dx': 0}),
    ('cab_combine_backward', {'dout': 0, 'ldo': 832, 'g': 0, 'x': 0, 'r': 0, 'gamma': 0, 'dtype': 2, 'dg': 0, 'dx': 0,
                              'dr': 0, 'dgamma': 0, 'n_pixels': 12, 'C': 256, 'accumulate_dx': 0}),
    ('cab_combine_backward', {'dout': 0, 'ldo': 832, 'g': 0, 'x': 0, 'r': 0, 'gamma': 0, 'dtype': 0, 'dg': 0, 'dx': 0,
                              'dr': 0, 'dgamma': 0, 'n_pixels': 12, 'C': 256, 'accumulate_dx': 0}),
    ('softmax_backward', {'p': 0, 'dp': 0, 'ds': 0, 'rows': 12, 'cols': 6, 'alpha': 0.08838834764831845}),
    ('conv_dgrad', {'dy': 0, 'lddy': 8, 'dtype': 0, 'w_packed': 0, 'w_dtype': 0, 'w_sco': 256, 'w_stap': 256, 'dx': 0,
                    'lddx': 256, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256, 'Cout': 8, 'KH': 1, 'KW': 1, 'stride': 1,
                    'pad': 0, 'OH': 2, 'OW': 3, 'accumulate': 0}),
    ('conv_dgrad', {'dy': 0, 'lddy': 144, 'dtype': 0, 'w_packed': 0, 'w_dtype': 0, 'w_sco': 48, 'w_stap': 48, 'dx': 0,
                    'lddx': 48, 'N': 2, 'H': 4, 'W': 6, 'Cin': 48, 'Cout': 144, 'KH': 1, 'KW': 1, 'stride': 1,
                    'pad': 0, 'OH': 4, 'OW': 6, 'accumulate': 1}),
    ('conv_dgrad', {'dy': 0, 'lddy': 256, 'dtype': 0, 'w_packed': 0, 'w_dtype': 0, 'w_sco': 7488, 'w_stap': 832,
                    'dx': 0, 'lddx': 832, 'N': 2, 'H': 2, 'W': 3, 'Cin': 832, 'Cout': 256, 'KH': 3, 'KW': 3,
                    'stride': 1, 'pad': 1, 'OH': 2, 'OW': 3, 'accumulate': 0}),
    ('conv_dgrad', {'dy': 0, 'lddy': 64, 'dtype': 0, 'w_packed': 0, 'w_dtype': 0, 'w_sco': 576, 'w_stap': 64, 'dx': 0,
                    'lddx': 64, 'N': 2, 'H': 16, 'W': 24, 'Cin': 64, 'Cout': 64, 'KH': 3, 'KW': 3, 'stride': 2,
                    'pad': 1, 'OH': 8, 'OW': 12, 'accumulate': 0}),
    ('conv_dgrad', {'dy': 0, 'lddy': 256, 'dtype': 0, 'w_packed': 0, 'w_dtype': 0, 'w_sco': 256, 'w_stap': 256,
                    'dx': 0, 'lddx': 832, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256, 'Cout': 256, 'KH': 1, 'KW': 1,
                    'stride': 1, 'pad': 0, 'OH': 2, 'OW': 3, 'accumulate': 1}),
    ('conv_dgrad', {'dy': 0, 'lddy': 256, 'dtype': 0, 'w_packed': 0, 'w_dtype': 0, 'w_sco': 5184, 'w_stap': 576,
                    'dx': 0, 'lddx': 832, 'N': 2, 'H': 2, 'W': 3, 'Cin': 576, 'Cout': 256, 'KH': 3, 'KW': 3,
                    'stride': 1, 'pad': 1, 'OH': 2, 'OW': 3, 'accumulate': 1}),
    ('conv_dgrad', {'dy': 0, 'lddy': 5, 'dtype': 0, 'w_packed': 0, 'w_dtype': 0, 'w_sco': 256, 'w_stap': 256, 'dx': 0,
                    'lddx': 256, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256, 'Cout': 5, 'KH': 1, 'KW': 1, 'stride': 1,
                    'pad': 0, 'OH': 8, 'OW': 16, 'accumulate': 0}),
    ('conv_wgrad', {'dy': 0, 'lddy': 8, 'dtype': 0, 'x': 0, 'x_dtype': 1, 'sxn': 1536, 'sxh': 768, 'sxw': 256,
                    'sxc': 1, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256, 'Cout': 8, 'KH': 1, 'KW': 1,
                    'stride': 1, 'pad': 0, 'OH': 2, 'OW': 3}),
    ('conv_wgrad', {'dy': 0, 'lddy': 5, 'dtype': 0, 'x': 0, 'x_dtype': 1, 'sxn': 32768, 'sxh': 4096, 'sxw': 256,
                    'sxc': 1, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256, 'Cout': 5, 'KH': 1, 'KW': 1,
                    'stride': 1, 'pad': 0, 'OH': 8, 'OW': 16}),
    ('conv_wgrad', {'dy': 0, 'lddy': 8, 'dtype': 0, 'x': 0, 'x_dtype': 2, 'sxn': 1536, 'sxh': 768, 'sxw': 256,
                    'sxc': 1, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256, 'Cout': 8, 'KH': 1, 'KW': 1,
                    'stride': 1, 'pad': 0, 'OH': 2, 'OW': 3}),
    ('conv_wgrad', {'dy': 0, 'lddy': 5, 'dtype': 0, 'x': 0, 'x_dtype': 2, 'sxn': 32768, 'sxh': 4096, 'sxw': 256,
                    'sxc': 1, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256, 'Cout': 5, 'KH': 1, 'KW': 1,
                    'stride': 1, 'pad': 0, 'OH': 8, 'OW': 16}),
    ('conv_wgrad', {'dy': 0, 'lddy': 8, 'dtype': 0, 'x': 0, 'x_dtype': 0, 'sxn': 1536, 'sxh': 768, 'sxw': 256,
                    'sxc': 1, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256, 'Cout': 8, 'KH': 1, 'KW': 1,
                    'stride': 1, 'pad': 0, 'OH': 2, 'OW': 3}),
    ('conv_wgrad', {'dy': 0, 'lddy': 256, 'dtype': 0, 'x': 0, 'x_dtype': 0, 'sxn': 4992, 'sxh': 2496, 'sxw': 832,
                    'sxc': 1, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 832, 'Cout': 256, 'KH': 3, 'KW': 3,
                    'stride': 1, 'pad': 1, 'OH': 2, 'OW': 3}),
    ('conv_wgrad', {'dy': 0, 'lddy': 64, 'dtype': 0, 'x': 0, 'x_dtype': 0, 'sxn': 24576, 'sxh': 1536, 'sxw': 64,
                    'sxc': 1, 'dw_oihw': 0, 'N': 2, 'H': 16, 'W': 24, 'Cin': 64, 'Cout': 64, 'KH': 3, 'KW': 3,
                    'stride': 2, 'pad': 1, 'OH': 8, 'OW': 12}),
    ('conv_wgrad', {'dy': 0, 'lddy': 16, 'dtype': 0, 'x': 0, 'x_dtype': 0, 'sxn': 18432, 'sxh': 96, 'sxw': 1,
                    'sxc': 6144, 'dw_oihw': 0, 'N': 2, 'H': 64, 'W': 96, 'Cin': 3, 'Cout': 16, 'KH': 3, 'KW': 3,
                    'stride': 2, 'pad': 1, 'OH': 32, 'OW': 48}),
    ('conv_wgrad', {'dy': 0, 'lddy': 64, 'dtype': 0, 'x': 0, 'x_dtype': 0, 'sxn': 18432, 'sxh': 96, 'sxw': 1,
                    'sxc': 6144, 'dw_oihw': 0, 'N': 2, 'H': 64, 'W': 96, 'Cin': 3, 'Cout': 64, 'KH': 7, 'KW': 7,
                    'stride': 2, 'pad': 3, 'OH': 32, 'OW': 48}),
    ('conv_wgrad', {'dy': 0, 'lddy': 256, 'dtype': 0, 'x': 0, 'x_dtype': 0, 'sxn': 4992, 'sxh': 2496, 'sxw': 832,
                    'sxc': 1, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256, 'Cout': 256, 'KH': 1, 'KW': 1,
                    'stride': 1, 'pad': 0, 'OH': 2, 'OW': 3}),
    ('conv_wgrad', {'dy': 0, 'lddy': 256, 'dtype': 0, 'x': 0, 'x_dtype': 0, 'sxn': 4992, 'sxh': 2496, 'sxw': 832,
                    'sxc': 1, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 576, 'Cout': 256, 'KH': 3, 'KW': 3,
                    'stride': 1, 'pad': 1, 'OH': 2, 'OW': 3}),
    ('conv_wgrad', {'dy': 0, 'lddy': 5, 'dtype': 0, 'x': 0, 'x_dtype': 0, 'sxn': 32768, 'sxh': 4096, 'sxw': 256,
                    'sxc': 1, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256, 'Cout': 5, 'KH': 1, 'KW': 1,
                    'stride': 1, 'pad': 0, 'OH': 8, 'OW': 16}),
    ('dwconv_dgrad', {'dy': 0, 'lddy': 16, 'dtype': 1, 'w_packed': 0, 'dx': 0, 'lddx': 16, 'N': 2, 'H': 32, 'W': 48,
                      'C': 16, 'k': 3, 'stride': 2, 'OH': 16, 'OW': 24, 'accumulate': 0}),
    ('dwconv_dgrad', {'dy': 0, 'lddy': 288, 'dtype': 1, 'w_packed': 0, 'dx': 0, 'lddx': 288, 'N': 2, 'H': 4, 'W': 6,
                      'C': 288, 'k': 5, 'stride': 2, 'OH': 2, 'OW': 3, 'accumulate': 0}),
    ('dwconv_dgrad', {'dy': 0, 'lddy': 16, 'dtype': 2, 'w_packed': 0, 'dx': 0, 'lddx': 16, 'N': 2, 'H': 32, 'W': 48,
                      'C': 16, 'k': 3, 'stride': 2, 'OH': 16, 'OW': 24, 'accumulate': 0}),
    ('dwconv_dgrad', {'dy': 0, 'lddy': 288, 'dtype': 2, 'w_packed': 0, 'dx': 0, 'lddx': 288, 'N': 2, 'H': 4, 'W': 6,
                      'C': 288, 'k': 5, 'stride': 2, 'OH': 2, 'OW': 3, 'accumulate': 0}),
    ('dwconv_dgrad', {'dy': 0, 'lddy': 256, 'dtype': 0, 'w_packed': 0, 'dx': 0, 'lddx': 256, 'N': 2, 'H': 2, 'W': 3,
                      'C': 256, 'k': 3, 'stride': 1, 'OH': 2, 'OW': 3, 'accumulate': 0}),
    ('dwconv_dgrad', {'dy': 0, 'lddy': 256, 'dtype': 0, 'w_packed': 0, 'dx': 0, 'lddx': 256, 'N': 2, 'H': 2, 'W': 3,
                      'C': 256, 'k': 3, 'stride': 1, 'OH': 2, 'OW': 3, 'accumulate': 1}),
    ('dwconv_dgrad', {'dy': 0, 'lddy': 120, 'dtype': 0, 'w_packed': 0, 'dx': 0, 'lddx': 120, 'N': 2, 'H': 4, 'W': 6,
                      'C': 120, 'k': 5, 'stride': 1, 'OH': 4, 'OW': 6, 'accumulate': 0}),
    ('dwconv_dgrad', {'dy': 0, 'lddy': 16, 'dtype': 0, 'w_packed': 0, 'dx': 0, 'lddx': 16, 'N': 2, 'H': 32, 'W': 48,
                      'C': 16, 'k': 3, 'stride': 2, 'OH': 16, 'OW': 24, 'accumulate': 0}),
    ('dwconv_dgrad', {'dy': 0, 'lddy': 288, 'dtype': 0, 'w_packed': 0, 'dx': 0, 'lddx': 288, 'N': 2, 'H': 4, 'W': 6,
                      'C': 288, 'k': 5, 'stride': 2, 'OH': 2, 'OW': 3, 'accumulate': 0}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 88, 'x': 0, 'ldx': 88, 'dtype': 1, 'dw': 0, 'N': 2, 'H': 8, 'W': 12, 'C': 88,
                      'k': 3, 'stride': 1, 'OH': 8, 'OW': 12}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 256, 'dtype': 1, 'dw': 0, 'N': 2, 'H': 2, 'W': 3, 'C': 256,
                      'k': 3, 'stride': 1, 'OH': 2, 'OW': 3}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 960, 'x': 0, 'ldx': 960, 'dtype': 1, 'dw': 0, 'N': 2, 'H': 8, 'W': 16, 'C': 960,
                      'k': 5, 'stride': 1, 'OH': 8, 'OW': 16}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 120, 'x': 0, 'ldx': 120, 'dtype': 1, 'dw': 0, 'N': 2, 'H': 4, 'W': 6, 'C': 120,
                      'k': 5, 'stride': 1, 'OH': 4, 'OW': 6}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 16, 'x': 0, 'ldx': 16, 'dtype': 1, 'dw': 0, 'N': 2, 'H': 32, 'W': 48, 'C': 16,
                      'k': 3, 'stride': 2, 'OH': 16, 'OW': 24}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 672, 'x': 0, 'ldx': 672, 'dtype': 1, 'dw': 0, 'N': 2, 'H': 16, 'W': 32,
                      'C': 672, 'k': 5, 'stride': 2, 'OH': 8, 'OW': 16}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 288, 'x': 0, 'ldx': 288, 'dtype': 1, 'dw': 0, 'N': 2, 'H': 4, 'W': 6, 'C': 288,
                      'k': 5, 'stride': 2, 'OH': 2, 'OW': 3}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 88, 'x': 0, 'ldx': 88, 'dtype': 2, 'dw': 0, 'N': 2, 'H': 8, 'W': 12, 'C': 88,
                      'k': 3, 'stride': 1, 'OH': 8, 'OW': 12}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 256, 'dtype': 2, 'dw': 0, 'N': 2, 'H': 2, 'W': 3, 'C': 256,
                      'k': 3, 'stride': 1, 'OH': 2, 'OW': 3}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 960, 'x': 0, 'ldx': 960, 'dtype': 2, 'dw': 0, 'N': 2, 'H': 8, 'W': 16, 'C': 960,
                      'k': 5, 'stride': 1, 'OH': 8, 'OW': 16}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 120, 'x': 0, 'ldx': 120, 'dtype': 2, 'dw': 0, 'N': 2, 'H': 4, 'W': 6, 'C': 120,
                      'k': 5, 'stride': 1, 'OH': 4, 'OW': 6}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 16, 'x': 0, 'ldx': 16, 'dtype': 2, 'dw': 0, 'N': 2, 'H': 32, 'W': 48, 'C': 16,
                      'k': 3, 'stride': 2, 'OH': 16, 'OW': 24}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 672, 'x': 0, 'ldx': 672, 'dtype': 2, 'dw': 0, 'N': 2, 'H': 16, 'W': 32,
                      'C': 672, 'k': 5, 'stride': 2, 'OH': 8, 'OW': 16}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 288, 'x': 0, 'ldx': 288, 'dtype': 2, 'dw': 0, 'N': 2, 'H': 4, 'W': 6, 'C': 288,
                      'k': 5, 'stride': 2, 'OH': 2, 'OW': 3}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 88, 'x': 0, 'ldx': 88, 'dtype': 0, 'dw': 0, 'N': 2, 'H': 8, 'W': 12, 'C': 88,
                      'k': 3, 'stride': 1, 'OH': 8, 'OW': 12}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 256, 'dtype': 0, 'dw': 0, 'N': 2, 'H': 2, 'W': 3, 'C': 256,
                      'k': 3, 'stride': 1, 'OH': 2, 'OW': 3}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 960, 'x': 0, 'ldx': 960, 'dtype': 0, 'dw': 0, 'N': 2, 'H': 8, 'W': 16, 'C': 960,
                      'k': 5, 'stride': 1, 'OH': 8, 'OW': 16}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 120, 'x': 0, 'ldx': 120, 'dtype': 0, 'dw': 0, 'N': 2, 'H': 4, 'W': 6, 'C': 120,
                      'k': 5, 'stride': 1, 'OH': 4, 'OW': 6}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 16, 'x': 0, 'ldx': 16, 'dtype': 0, 'dw': 0, 'N': 2, 'H': 32, 'W': 48, 'C': 16,
                      'k': 3, 'stride': 2, 'OH': 16, 'OW': 24}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 672, 'x': 0, 'ldx': 672, 'dtype': 0, 'dw': 0, 'N': 2, 'H': 16, 'W': 32,
                      'C': 672, 'k': 5, 'stride': 2, 'OH': 8, 'OW': 16}),
    ('dwconv_wgrad', {'dy': 0, 'lddy': 288, 'x': 0, 'ldx': 288, 'dtype': 0, 'dw': 0, 'N': 2, 'H': 4, 'W': 6, 'C': 288,
                      'k': 5, 'stride': 2, 'OH': 2, 'OW': 3}),
    ('resample_sep', {'in': 0, 'in_dtype': 1, 'isn': 3840, 'isy': 1920, 'isx': 640, 'isc': 1, 'out': 0, 'out_dtype': 1,
                      'osn': 128, 'osy': 128, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 1, 'OW': 1, 'C': 128,
                      'accumulate': 0, 'y_op': ('bilinear', 1, 2, True), 'x_op': ('bilinear', 1, 3, True)}),
    ('resample_sep', {'in': 0, 'in_dtype': 1, 'isn': 1152, 'isy': 384, 'isx': 128, 'isc': 1, 'out': 0, 'out_dtype': 1,
                      'osn': 3840, 'osy': 1920, 'osx': 640, 'osc': 1, 'N': 2, 'OH': 2, 'OW': 3, 'C': 128,
                      'accumulate': 0, 'y_op': ('bilinear', 3, 2, False), 'x_op': ('bilinear', 3, 3, False)}),
    ('resample_sep', {'in': 0, 'in_dtype': 1, 'isn': 768, 'isy': 384, 'isx': 128, 'isc': 1, 'out': 0, 'out_dtype': 1,
                      'osn': 128, 'osy': 128, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 1, 'OW': 1, 'C': 128,
                      'accumulate': 0, 'y_op': ('pool', 2, 1, False), 'x_op': ('pool', 3, 1, False)}),
    ('resample_sep', {'in': 0, 'in_dtype': 1, 'isn': 1152, 'isy': 384, 'isx': 128, 'isc': 1, 'out': 0, 'out_dtype': 1,
                      'osn': 768, 'osy': 384, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 2, 'OW': 3, 'C': 128,
                      'accumulate': 1, 'y_op': ('pool', 2, 3, True), 'x_op': ('pool', 3, 3, True)}),
    ('resample_sep', {'in': 0, 'in_dtype': 1, 'isn': 3840, 'isy': 1920, 'isx': 640, 'isc': 1, 'out': 0, 'out_dtype': 1,
                      'osn': 1152, 'osy': 384, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 3, 'OW': 3, 'C': 128,
                      'accumulate': 4, 'y_op': ('bilinear', 3, 2, True), 'x_op': ('bilinear', 3, 3, True)}),
    ('resample_sep', {'in': 0, 'in_dtype': 1, 'isn': 128, 'isy': 128, 'isx': 128, 'isc': 1, 'out': 0, 'out_dtype': 1,
                      'osn': 3840, 'osy': 1920, 'osx': 640, 'osc': 1, 'N': 2, 'OH': 2, 'OW': 3, 'C': 128,
                      'accumulate': 4, 'y_op': ('bilinear', 1, 2, False), 'x_op': ('bilinear', 1, 3, False)}),
    ('resample_sep', {'in': 0, 'in_dtype': 1, 'isn': 768, 'isy': 384, 'isx': 128, 'isc': 1, 'out': 0, 'out_dtype': 1,
                      'osn': 1152, 'osy': 384, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 3, 'OW': 3, 'C': 128,
                      'accumulate': 4, 'y_op': ('pool', 2, 3, False), 'x_op': ('pool', 3, 3, False)}),
    ('resample_sep', {'in': 0, 'in_dtype': 1, 'isn': 128, 'isy': 128, 'isx': 128, 'isc': 1, 'out': 0, 'out_dtype': 1,
                      'osn': 768, 'osy': 384, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 2, 'OW': 3, 'C': 128,
                      'accumulate': 5, 'y_op': ('pool', 2, 1, True), 'x_op': ('pool', 3, 1, True)}),
    ('resample_sep', {'in': 0, 'in_dtype': 1, 'isn': 81920, 'isy': 10240, 'isx': 640, 'isc': 1, 'out': 0,
                      'out_dtype': 0, 'osn': 1024, 'osy': 128, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 8, 'OW': 1,
                      'C': 128, 'accumulate': 0, 'y_op': ('identity', 8, 8, False),
                      'x_op': ('bilinear', 1, 16, True)}),
    ('resample_sep', {'in': 0, 'in_dtype': 1, 'isn': 16384, 'isy': 2048, 'isx': 128, 'isc': 1, 'out': 0,
                      'out_dtype': 0, 'osn': 1024, 'osy': 128, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 8, 'OW': 1,
                      'C': 128, 'accumulate': 0, 'y_op': ('identity', 8, 8, False), 'x_op': ('pool', 16, 1, False)}),
    ('resample_sep', {'in': 0, 'in_dtype': 2, 'isn': 3840, 'isy': 1920, 'isx': 640, 'isc': 1, 'out': 0, 'out_dtype': 2,
                      'osn': 128, 'osy': 128, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 1, 'OW': 1, 'C': 128,
                      'accumulate': 0, 'y_op': ('bilinear', 1, 2, True), 'x_op': ('bilinear', 1, 3, True)}),
    ('resample_sep', {'in': 0, 'in_dtype': 2, 'isn': 1152, 'isy': 384, 'isx': 128, 'isc': 1, 'out': 0, 'out_dtype': 2,
                      'osn': 3840, 'osy': 1920, 'osx': 640, 'osc': 1, 'N': 2, 'OH': 2, 'OW': 3, 'C': 128,
                      'accumulate': 0, 'y_op': ('bilinear', 3, 2, False), 'x_op': ('bilinear', 3, 3, False)}),
    ('resample_sep', {'in': 0, 'in_dtype': 2, 'isn': 768, 'isy': 384, 'isx': 128, 'isc': 1, 'out': 0, 'out_dtype': 2,
                      'osn': 128, 'osy': 128, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 1, 'OW': 1, 'C': 128,
                      'accumulate': 0, 'y_op': ('pool', 2, 1, False), 'x_op': ('pool', 3, 1, False)}),
    ('resample_sep', {'in': 0, 'in_dtype': 2, 'isn': 1152, 'isy': 384, 'isx': 128, 'isc': 1, 'out': 0, 'out_dtype': 2,
                      'osn': 768, 'osy': 384, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 2, 'OW': 3, 'C': 128,
                      'accumulate': 1, 'y_op': ('pool', 2, 3, True), 'x_op': ('pool', 3, 3, True)}),
    ('resample_sep', {'in': 0, 'in_dtype': 2, 'isn': 3840, 'isy': 1920, 'isx': 640, 'isc': 1, 'out': 0, 'out_dtype': 2,
                      'osn': 1152, 'osy': 384, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 3, 'OW': 3, 'C': 128,
                      'accumulate': 4, 'y_op': ('bilinear', 3, 2, True), 'x_op': ('bilinear', 3, 3, True)}),
    ('resample_sep', {'in': 0, 'in_dtype': 2, 'isn': 128, 'isy': 128, 'isx': 128, 'isc': 1, 'out': 0, 'out_dtype': 2,
                      'osn': 3840, 'osy': 1920, 'osx': 640, 'osc': 1, 'N': 2, 'OH': 2, 'OW': 3, 'C': 128,
                      'accumulate': 4, 'y_op': ('bilinear', 1, 2, False), 'x_op': ('bilinear', 1, 3, False)}),
    ('resample_sep', {'in': 0, 'in_dtype': 2, 'isn': 768, 'isy': 384, 'isx': 128, 'isc': 1, 'out': 0, 'out_dtype': 2,
                      'osn': 1152, 'osy': 384, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 3, 'OW': 3, 'C': 128,
                      'accumulate': 4, 'y_op': ('pool', 2, 3, False), 'x_op': ('pool', 3, 3, False)}),
    ('resample_sep', {'in': 0, 'in_dtype': 2, 'isn': 128, 'isy': 128, 'isx': 128, 'isc': 1, 'out': 0, 'out_dtype': 2,
                      'osn': 768, 'osy': 384, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 2, 'OW': 3, 'C': 128,
                      'accumulate': 5, 'y_op': ('pool', 2, 1, True), 'x_op': ('pool', 3, 1, True)}),
    ('resample_sep', {'in': 0, 'in_dtype': 2, 'isn': 81920, 'isy': 10240, 'isx': 640, 'isc': 1, 'out': 0,
                      'out_dtype': 0, 'osn': 1024, 'osy': 128, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 8, 'OW': 1,
                      'C': 128, 'accumulate': 0, 'y_op': ('identity', 8, 8, False),
                      'x_op': ('bilinear', 1, 16, True)}),
    ('resample_sep', {'in': 0, 'in_dtype': 2, 'isn': 16384, 'isy': 2048, 'isx': 128, 'isc': 1, 'out': 0,
                      'out_dtype': 0, 'osn': 1024, 'osy': 128, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 8, 'OW': 1,
                      'C': 128, 'accumulate': 0, 'y_op': ('identity', 8, 8, False), 'x_op': ('pool', 16, 1, False)}),
    ('resample_sep', {'in': 0, 'in_dtype': 0, 'isn': 1024, 'isy': 128, 'isx': 128, 'isc': 1, 'out': 0, 'out_dtype': 1,
                      'osn': 128, 'osy': 128, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 1, 'OW': 1, 'C': 128,
                      'accumulate': 0, 'y_op': ('pool', 8, 1, False), 'x_op': ('identity', 1, 1, False)}),
    ('resample_sep', {'in': 0, 'in_dtype': 0, 'isn': 1024, 'isy': 128, 'isx': 128, 'isc': 1, 'out': 0, 'out_dtype': 2,
                      'osn': 128, 'osy': 128, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 1, 'OW': 1, 'C': 128,
                      'accumulate': 0, 'y_op': ('pool', 8, 1, False), 'x_op': ('identity', 1, 1, False)}),
    ('resample_sep', {'in': 0, 'in_dtype': 0, 'isn': 10240, 'isy': 320, 'isx': 5, 'isc': 1, 'out': 0, 'out_dtype': 0,
                      'osn': 640, 'osy': 80, 'osx': 5, 'osc': 1, 'N': 2, 'OH': 8, 'OW': 16, 'C': 5, 'accumulate': 0,
                      'y_op': ('bilinear', 8, 32, True), 'x_op': ('bilinear', 16, 64, True)}),
    ('resample_sep', {'in': 0, 'in_dtype': 0, 'isn': 3840, 'isy': 1920, 'isx': 640, 'isc': 1, 'out': 0, 'out_dtype': 0,
                      'osn': 128, 'osy': 128, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 1, 'OW': 1, 'C': 128,
                      'accumulate': 0, 'y_op': ('bilinear', 1, 2, True), 'x_op': ('bilinear', 1, 3, True)}),
    ('resample_sep', {'in': 0, 'in_dtype': 0, 'isn': 1152, 'isy': 384, 'isx': 128, 'isc': 1, 'out': 0, 'out_dtype': 0,
                      'osn': 3840, 'osy': 1920, 'osx': 640, 'osc': 1, 'N': 2, 'OH': 2, 'OW': 3, 'C': 128,
                      'accumulate': 0, 'y_op': ('bilinear', 3, 2, False), 'x_op': ('bilinear', 3, 3, False)}),
    ('resample_sep', {'in': 0, 'in_dtype': 0, 'isn': 768, 'isy': 96, 'isx': 8, 'isc': 1, 'out': 0, 'out_dtype': 0,
                      'osn': 48, 'osy': 24, 'osx': 8, 'osc': 1, 'N': 2, 'OH': 2, 'OW': 3, 'C': 8, 'accumulate': 0,
                      'y_op': ('bilinear', 2, 8, True), 'x_op': ('bilinear', 3, 12, True)}),
    ('resample_sep', {'in': 0, 'in_dtype': 0, 'isn': 1152, 'isy': 384, 'isx': 128, 'isc': 1, 'out': 0, 'out_dtype': 0,
                      'osn': 768, 'osy': 384, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 2, 'OW': 3, 'C': 128,
                      'accumulate': 1, 'y_op': ('pool', 2, 3, True), 'x_op': ('pool', 3, 3, True)}),
    ('resample_sep', {'in': 0, 'in_dtype': 0, 'isn': 49152, 'isy': 96, 'isx': 1, 'isc': 6144, 'out': 0, 'out_dtype': 0,
                      'osn': 768, 'osy': 96, 'osx': 8, 'osc': 1, 'N': 2, 'OH': 8, 'OW': 12, 'C': 8, 'accumulate': 2,
                      'y_op': ('bilinear', 8, 64, True), 'x_op': ('bilinear', 12, 96, True)}),
    ('resample_sep', {'in': 0, 'in_dtype': 0, 'isn': 640, 'isy': 80, 'isx': 5, 'isc': 1, 'out': 0, 'out_dtype': 0,
                      'osn': 10240, 'osy': 320, 'osx': 5, 'osc': 1, 'N': 2, 'OH': 32, 'OW': 64, 'C': 5,
                      'accumulate': 4, 'y_op': ('bilinear', 8, 32, False), 'x_op': ('bilinear', 16, 64, False)}),
    ('resample_sep', {'in': 0, 'in_dtype': 0, 'isn': 3840, 'isy': 1920, 'isx': 640, 'isc': 1, 'out': 0, 'out_dtype': 0,
                      'osn': 1152, 'osy': 384, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 3, 'OW': 3, 'C': 128,
                      'accumulate': 4, 'y_op': ('bilinear', 3, 2, True), 'x_op': ('bilinear', 3, 3, True)}),
    ('resample_sep', {'in': 0, 'in_dtype': 0, 'isn': 128, 'isy': 128, 'isx': 128, 'isc': 1, 'out': 0, 'out_dtype': 0,
                      'osn': 3840, 'osy': 1920, 'osx': 640, 'osc': 1, 'N': 2, 'OH': 2, 'OW': 3, 'C': 128,
                      'accumulate': 4, 'y_op': ('bilinear', 1, 2, False), 'x_op': ('bilinear', 1, 3, False)}),
    ('resample_sep', {'in': 0, 'in_dtype': 0, 'isn': 48, 'isy': 24, 'isx': 8, 'isc': 1, 'out': 0, 'out_dtype': 0,
                      'osn': 768, 'osy': 96, 'osx': 8, 'osc': 1, 'N': 2, 'OH': 8, 'OW': 12, 'C': 8, 'accumulate': 4,
                      'y_op': ('bilinear', 2, 8, False), 'x_op': ('bilinear', 3, 12, False)}),
    ('resample_sep', {'in': 0, 'in_dtype': 0, 'isn': 128, 'isy': 128, 'isx': 128, 'isc': 1, 'out': 0, 'out_dtype': 0,
                      'osn': 768, 'osy': 384, 'osx': 128, 'osc': 1, 'N': 2, 'OH': 2, 'OW': 3, 'C': 128,
                      'accumulate': 5, 'y_op': ('pool', 2, 1, True), 'x_op': ('pool', 3, 1, True)}),
    ('channel_sum', {'x': 0, 'ldx': 288, 'dtype': 1, 'N': 2, 'HW': 6, 'C': 288, 'out': 0, 'scratch_bytes': 147968}),
    ('channel_sum', {'x': 0, 'ldx': 288, 'dtype': 2, 'N': 2, 'HW': 6, 'C': 288, 'out': 0, 'scratch_bytes': 147968}),
    ('channel_sum', {'x': 0, 'ldx': 288, 'dtype': 0, 'N': 2, 'HW': 6, 'C': 288, 'out': 0, 'scratch_bytes': 147968}),
]


def _launch(lib, k, call, what):
    for op in k.ops:
        op.reset()
    check(call(), what)
    torch.cuda.synchronize()
    for op in k.ops:
        op.check_canaries(what)
    return [op.buf.clone() for op in k.ops if op.out]


@pytest.mark.parametrize("entry,a", [pytest.param(e, a, id=variant_key(e, a).replace(" ", "_")) for e, a in CASES])
def test_variant_against_float64(entry, a):
    lib = _lib.load()
    k = Case()
    call = RUNNERS[entry](lib, a, k)
    first = _launch(lib, k, call, entry)
    for name, op, ref, tol in k.checks:
        compare(f"{entry} {name}", op, ref, tol)
    again = _launch(lib, k, call, entry)
    for b0, b1 in zip(first, again):
        assert torch.equal(b0.view(ITD[b0.dtype]), b1.view(ITD[b1.dtype])), f"{entry}: not bit-reproducible"
    if "rt" in variant_key(entry, a).split():
        old = lib.cabinet_debug_flags(0)
        try:
            lib.cabinet_debug_flags(old | 128)   # the register-fed reduction instead of the shared-memory-staged one
            _launch(lib, k, call, entry + " (register-fed)")
        finally:
            lib.cabinet_debug_flags(old)
        for name, op, ref, tol in k.checks:
            compare(f"{entry} {name} (register-fed)", op, ref, tol)
