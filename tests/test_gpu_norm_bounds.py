"""LayerNorm, column-sum, LayerScale-backward, scale_cols / add / cast and depth-wise convolution kernels against fp64
with elementwise bounds (tests/norm_ref.py), in every template instantiation the launchers can pick, in both dtypes.
Every case calls the C ABI with each output inside a NaN-filled buffer (nothing outside the outputs may change),
asserts from the torch.profiler trace which instantiation ran with which grid (the launchers' arithmetic in
norm_ref), runs every backward twice (the results must be bit-identical) and prints its largest err / bound ratio."""
import ctypes
import time

import pytest
import torch

import norm_ref as NR
import tc_ref as R
from adaptersis_b200 import _lib
from adaptersis_b200._lib import ptr
from tc_ref import bits, guarded, guards_intact

pytestmark = pytest.mark.gpu
DEV = "cuda"
BF, F32 = torch.bfloat16, torch.float32
DTS = (F32, BF)
VT = {F32: "float", BF: "__nv_bfloat16"}
TAG = {F32: "f32", BF: "bf16"}
EPS = 1e-6


# ------------------------------------------------------------------------------------------- the launch plans
def _cdiv(a, b):
    return -(-a // b)


def reduce_plan(nparts, ncols):
    return (f"reduce_partials_kernel<{NR.reduce_pl(nparts)}>", (_cdiv(ncols, 32),))


def ln_fwd_plan(xt, yt, R_, C):
    return [(f"ln_fwd_kernel<{VT[xt]},{VT[yt]},{NR.ln_nv(C)}>", (NR.ln_fwd_grid(R_),))]


def ln_bwd_plan(dt, xt, R_, C, want_g, want_b):
    grid = NR.ln_bwd_grid(R_)
    plan = [(f"ln_bwd2_kernel<{VT[dt]},{VT[xt]}>", (grid,))]
    if want_g or want_b:
        plan.append(reduce_plan(grid, 2 * C if (want_g and want_b) else C))
    return plan


def colsum_plan(xt, yt, M, N):
    rb = NR.colsum_rb(M, N)
    name = f"colsum_kernel<{VT[xt]},{VT[yt]},1>" if yt is not None else f"colsum_kernel<{VT[xt]},float,0>"
    return [(name, (_cdiv(N, 128), rb)), reduce_plan(rb, N)]


def layerscale_plan(ut, M, N, want_g, want_b):
    rb = NR.colsum_rb(M)
    return [(f"layerscale_bwd_kernel<{VT[ut]}>", (_cdiv(N, 128), rb)),
            reduce_plan(rb, 2 * N if (want_g and want_b) else N)]


def dwconv_fwd_plan(t, B, ntok, C):
    return [(f"dwconv_fwd_kernel<{VT[t]}>", (NR.dwconv_fwd_grid(B, ntok, C),))]


def dwconv_bwd_plan(t, B, ntok, C, fuse):
    plan = [(f"dwconv_gelu_grad_kernel<{VT[t]}>", (_cdiv(B * ntok * C // 4, 256),))] if fuse else []
    plan.append((f"dwconv_bwd_kernel<{VT[t]}>", (_cdiv(C, 128), NR.dwconv_row_blocks(B * ntok, C))))
    plan.append(("dwconv_reduce_kernel", (_cdiv(10 * C, 256),)))
    return plan


def _norm(name):
    return name.replace(" ", "").replace("(bool)", "").replace("true", "1").replace("false", "0")


def expect_launches(ks, plan):
    """The trace holds exactly the planned launches, in order, with their instantiations and grids."""
    assert len(ks) == len(plan), f"expected {[p[0] for p in plan]}, trace has {[k[0] for k in ks]}"
    for (name, grid), (want, wgrid) in zip(ks, plan):
        assert _norm("asis::" + want + "(") in _norm(name), (name, want)
        assert tuple(grid) + (1,) * (3 - len(grid)) == tuple(wgrid) + (1,) * (3 - len(wgrid)), (name, grid, wgrid)


def run_traced(fn, plan):
    r, ks = R.traced(fn)
    expect_launches(ks, plan)
    return r


def report(tag, reps, t0):
    worst = max(reps, key=lambda r: r.ratio)
    print(f"[{tag}] max err/bound {worst.ratio:.3g} ({worst.name} at {worst.where}) [{time.time() - t0:.1f} s]")
    for r in reps:
        assert r.ok, f"[{tag}] {r}"


def intact(bufs, tag):
    assert all(guards_intact(b) for b in bufs), f"[{tag}] a kernel wrote outside its output"


def same_bits(a, b):
    return all(torch.equal(bits(x), bits(y)) for x, y in zip(a, b) if x is not None)


def lib():
    return _lib.load()


def gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


# ------------------------------------------------------------------------------------------ LayerNorm forward
NV_CS = {1: (4, 68, 128), 2: (132, 256), 3: (260, 384), 4: (388, 512), 6: (516, 640, 768), 8: (772, 1020, 1024)}
LN_FWD = [(xt, yt, nv) for xt in DTS for yt in DTS for nv in NV_CS]


def ln_fwd_rows(R_, C, xt, g):
    """randn * 2 + 0.5, with (R >= 7) a constant row, a zero row, a row of std 1e-3, a row at mean offset 1e3 (f32 x)
    and a row with one large outlier."""
    x = torch.randn(R_, C, device=DEV, generator=g) * 2 + 0.5
    if R_ >= 7:
        x[0] = 0.7
        x[1] = 0.0
        x[2] = 0.5 + 1e-3 * torch.randn(C, device=DEV, generator=g)
        if xt == F32:
            x[3] = 1e3 + torch.randn(C, device=DEV, generator=g)
        x[4, C // 2] = 500.0
    return x.to(xt)


def abi_ln_fwd(x, g, b, yt, stats):
    R_, C = x.shape
    by, y = guarded((R_, C), yt)
    bm, mean = guarded((R_,), F32)
    br, rstd = guarded((R_,), F32)
    _lib.check(lib().asis_layernorm_forward(ptr(x), _lib.dt(x), ptr(g), ptr(b), ptr(y), _lib.dt(y),
                                            ptr(mean) if stats else None, ptr(rstd) if stats else None, R_, C, EPS,
                                            _lib.stream()))
    return y, mean, rstd, [by, bm, br]


@pytest.mark.parametrize("xt,yt,nv", LN_FWD, ids=[f"{TAG[a]}-{TAG[b]}-NV{n}" for a, b, n in LN_FWD])
def test_ln_fwd(xt, yt, nv):
    t0 = time.time()
    g = gen(nv)
    reps = []
    shapes = [(R_, C) for C in NV_CS[nv] for R_ in (1, 7, 8 * 37 + 3)] + [(21180, NV_CS[nv][-1])]
    for R_, C in shapes:
        x = ln_fwd_rows(R_, C, xt, g)
        gm = torch.randn(C, device=DEV, generator=g)
        bt = torch.randn(C, device=DEV, generator=g)
        stats = R_ > 1                              # R = 1 runs the path without mean / rstd outputs
        y, mean, rstd, bufs = run_traced(lambda: abi_ln_fwd(x, gm, bt, yt, stats), ln_fwd_plan(xt, yt, R_, C))
        intact(bufs, f"ln_fwd R={R_} C={C}")
        refs = NR.ln_fwd_ref(x, gm, bt, EPS, nv)
        reps.append(R.check(f"y R={R_} C={C}", y, refs["y"][0], R.u_out(yt), refs["y"][1], block=NR.row_slabs(8)))
        if stats:
            for k, o in (("mean", mean), ("rstd", rstd)):
                reps.append(R.check(f"{k} R={R_} C={C}", o, refs[k][0], R.U_F32, refs[k][1], block=NR.row_slabs(8)))
        else:
            assert bool((bits(mean) == R.NAN_BITS[4]).all()) and bool((bits(rstd) == R.NAN_BITS[4]).all())
    report(f"ln_fwd {TAG[xt]}->{TAG[yt]} NV={nv}", reps, t0)


# ----------------------------------------------------------------------------------------- LayerNorm backward
LN_BWD = [(dt, xt, dres) for dt in DTS for xt in DTS for dres in (False, True)]
# (R, C, dgamma, dbeta, accumulate)
LN_BWD_SHAPES = [(3, 132, True, True, False), (95, 132, True, True, True), (95, 260, True, False, False),
                 (95, 260, False, True, True), (95, 260, False, False, False), (21180, 1024, True, True, False)]


def ln_bwd_inputs(R_, C, dt, xt, g):
    x = (torch.randn(R_, C, device=DEV, generator=g) * 2 + 0.5).to(xt)
    dy = torch.randn(R_, C, device=DEV, generator=g).to(dt)
    gm = torch.randn(C, device=DEV, generator=g)
    xf = x.float()
    mu = xf.mean(1)
    rs = torch.rsqrt(xf.var(1, unbiased=False) + EPS)
    dres = torch.randn(R_, C, device=DEV, generator=g)
    prior = (torch.randn(C, device=DEV, generator=g), torch.randn(C, device=DEV, generator=g))
    return dy, x, gm, mu, rs, dres, prior


def abi_ln_bwd(dy, x, gm, mu, rs, dres, want_g, want_b, prior):
    R_, C = x.shape
    bx, dx = guarded((R_, C), F32)
    bg, dg = guarded((C,), F32)
    bb, db = guarded((C,), F32)
    if prior is not None:
        dg.copy_(prior[0])
        db.copy_(prior[1])
    nbytes = lib().asis_layernorm_backward_workspace_bytes(R_, C)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    _lib.check(lib().asis_layernorm_backward(ptr(dy), _lib.dt(dy), ptr(x), _lib.dt(x), ptr(gm), ptr(mu), ptr(rs),
                                             ptr(dres), ptr(dx), ptr(dg) if want_g else None,
                                             ptr(db) if want_b else None, int(prior is not None), R_, C, ptr(ws),
                                             nbytes, _lib.stream()))
    return (dx, dg if want_g else None, db if want_b else None), [bx, bg, bb], (dg, db)


def ln_bwd_case(tag, dt, xt, use_dres, R_, C, want_g, want_b, acc, seed):
    t0 = time.time()
    dy, x, gm, mu, rs, dres, prior = ln_bwd_inputs(R_, C, dt, xt, gen(seed))
    dres = dres if use_dres else None
    prior = prior if acc else None
    args = (dy, x, gm, mu, rs, dres, want_g, want_b, prior)
    outs, bufs, (dg, db) = run_traced(lambda: abi_ln_bwd(*args), ln_bwd_plan(dt, xt, R_, C, want_g, want_b))
    intact(bufs, tag)
    for want, o in ((want_g, dg), (want_b, db)):       # a gradient not asked for stays untouched
        if not want:
            assert torch.equal(bits(o), bits(prior[0 if o is dg else 1])) if acc else \
                bool((bits(o) == R.NAN_BITS[4]).all()), f"[{tag}] an output not asked for was written"
    again, _, _ = abi_ln_bwd(*args)
    assert same_bits(outs, again), f"[{tag}] the backward is not run-to-run identical"
    pg, pb = prior if acc else (None, None)
    refs = NR.ln_bwd_ref(dy, x, gm, mu, rs, dres, NR.ln_bwd_grid(R_), pg, pb)
    reps = [R.check("dx", outs[0], refs["dx"][0], R.U_F32, refs["dx"][1], block=NR.row_slabs(2))]
    for k, o in (("dgamma", outs[1]), ("dbeta", outs[2])):
        if o is not None:
            reps.append(R.check(k, o, refs[k][0], R.U_F32, refs[k][1], block=NR.col_slabs))
    del refs
    report(tag, reps, t0)


@pytest.mark.parametrize("dt,xt,dres", LN_BWD, ids=[f"dy{TAG[a]}-x{TAG[b]}-{'dres' if r else 'nores'}"
                                                   for a, b, r in LN_BWD])
def test_ln_bwd(dt, xt, dres):
    for i, (R_, C, wg, wb, acc) in enumerate(LN_BWD_SHAPES):
        ln_bwd_case(f"ln_bwd dy={TAG[dt]} x={TAG[xt]} dres={dres} R={R_} C={C} dgamma={wg} dbeta={wb} acc={acc}",
                    dt, xt, dres, R_, C, wg, wb, acc, seed=i)


def test_ln_bwd_persistent():
    """[83388 x 1024], the adapters' largest LayerNorm: every block runs ~70 iterations, 592 partials (PL = 32)."""
    ln_bwd_case("ln_bwd persistent 83388 x 1024", BF, BF, True, 83388, 1024, True, True, False, seed=9)


# ------------------------------------------------------------------------------------------------ column sums
COLSUM = [(xt, yt) for xt in DTS for yt in DTS + (None,)]
# (M, N, ld, column offset, accumulate)
COLSUM_SHAPES = [(83388, 64, 64, 0, False), (37, 4, 4, 0, False), (1001, 132, 148, 8, False),
                 (3000, 1024, 1024, 0, True)]


def abi_colsum(X, Y, off, N, ld, prior):
    M = X.shape[0]
    bo, out = guarded((N,), F32)
    if prior is not None:
        out.copy_(prior)
    nbytes = lib().asis_colsum_workspace_bytes(M, N)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    xp = X.data_ptr() + off * X.element_size()
    yp = None if Y is None else Y.data_ptr() + off * Y.element_size()
    _lib.check(lib().asis_colsum(xp, _lib.dt(X), yp, _lib.dt(Y) if Y is not None else 0, ld, ptr(out),
                                 int(prior is not None), M, N, ptr(ws), nbytes, _lib.stream()))
    return out, [bo]


@pytest.mark.parametrize("xt,yt", COLSUM, ids=[f"{TAG[a]}-{TAG[b] if b else 'noY'}" for a, b in COLSUM])
def test_colsum(xt, yt):
    t0 = time.time()
    g = gen(5)
    reps = []
    for M, N, ld, off, acc in COLSUM_SHAPES:
        X = (torch.randn(M, ld, device=DEV, generator=g) + 0.25).to(xt)
        Y = None if yt is None else torch.randn(M, ld, device=DEV, generator=g).to(yt)
        prior = torch.randn(N, device=DEV, generator=g) if acc else None
        out, bufs = run_traced(lambda: abi_colsum(X, Y, off, N, ld, prior), colsum_plan(xt, yt, M, N))
        intact(bufs, f"colsum M={M} N={N}")
        ref, terms = NR.colsum_ref(X[:, off:off + N], None if Y is None else Y[:, off:off + N], prior=prior)
        reps.append(R.check(f"colsum M={M} N={N} ld={ld}", out, ref, R.U_F32, terms, block=NR.col_slabs))
    report(f"colsum {TAG[xt]} x {TAG[yt] if yt else '-'}", reps, t0)


# ------------------------------------------------------------------------------------------ LayerScale backward
LAYERSCALE = [(ut, mode) for ut in DTS for mode in ("both", "dgamma", "dbias")]


def abi_layerscale(d, u, gm, ut, want_g, want_b):
    M, N = d.shape
    bu, du = guarded((M, N), ut)
    bg, dg = guarded((N,), F32)
    bb, db = guarded((N,), F32)
    nbytes = lib().asis_layerscale_backward_workspace_bytes(M, N)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    _lib.check(lib().asis_layerscale_backward(ptr(d), ptr(u) if want_g else None, ptr(gm), ptr(du), _lib.dt(du),
                                              ptr(dg) if want_g else None, ptr(db) if want_b else None, M, N,
                                              ptr(ws), nbytes, _lib.stream()))
    return (du, dg if want_g else None, db if want_b else None), [bu, bg, bb], (dg, db)


@pytest.mark.parametrize("ut,mode", LAYERSCALE, ids=[f"{TAG[a]}-{m}" for a, m in LAYERSCALE])
def test_layerscale_bwd(ut, mode):
    t0 = time.time()
    g = gen(6)
    want_g, want_b = mode in ("both", "dgamma"), mode in ("both", "dbias")
    reps = []
    for M, N in ((21180, 1024), (1001, 196)):
        d = torch.randn(M, N, device=DEV, generator=g)
        u = torch.randn(M, N, device=DEV, generator=g).to(ut)
        gm = torch.randn(N, device=DEV, generator=g) * 0.1
        tag = f"layerscale {TAG[ut]} {mode} M={M} N={N}"
        outs, bufs, (dg, db) = run_traced(lambda: abi_layerscale(d, u, gm, ut, want_g, want_b),
                                          layerscale_plan(ut, M, N, want_g, want_b))
        intact(bufs, tag)
        for want, o in ((want_g, dg), (want_b, db)):
            assert want or bool((bits(o) == R.NAN_BITS[4]).all()), f"[{tag}] an output not asked for was written"
        again, _, _ = abi_layerscale(d, u, gm, ut, want_g, want_b)
        assert same_bits(outs, again), f"[{tag}] not run-to-run identical"
        refs = NR.layerscale_ref(d, u if want_g else None, gm, ut)
        assert torch.equal(bits(outs[0]), bits(refs["du"])), f"[{tag}] du differs from (d * gamma).to(UT)"
        if want_g:
            reps.append(R.check(f"dgamma M={M} N={N}", outs[1], refs["dgamma"][0], R.U_F32, refs["dgamma"][1],
                                block=NR.col_slabs))
        if want_b:
            reps.append(R.check(f"dbias M={M} N={N}", outs[2], refs["dbias"][0], R.U_F32, refs["dbias"][1],
                                block=NR.col_slabs))
    report(f"layerscale {TAG[ut]} {mode}", reps, t0)


# ------------------------------------------------------------------------------------- scale_cols / add / cast
ELEMENTWISE = ([("scale_cols", a, None, o) for a in DTS for o in DTS] +
               [("add", a, b, o) for a in DTS for b in DTS for o in DTS] +
               [("cast", a, None, o) for a in DTS for o in DTS])


def elementwise_plan(op, at, bt, ot, n):
    if op == "scale_cols":
        return [(f"scale_cols_kernel<{VT[at]},{VT[ot]}>", (_cdiv(n // 4, 256),))]
    if op == "add":
        return [(f"add_cast_kernel<{VT[at]},{VT[bt]},{VT[ot]},1>", (_cdiv(_cdiv(n, 4), 256),))]
    return [(f"add_cast_kernel<{VT[at]},{VT[at]},{VT[ot]},0>", (_cdiv(_cdiv(n, 4), 256),))]


@pytest.mark.parametrize("op,at,bt,ot", ELEMENTWISE,
                         ids=[f"{op}-{TAG[a]}-{TAG[b] if b else ''}-{TAG[o]}" for op, a, b, o in ELEMENTWISE])
def test_scale_add_cast_bit_exact(op, at, bt, ot):
    """One fp32 operation and the store: bit for bit against torch; n = 100003 leaves a scalar tail of 3."""
    g = gen(7)
    M, N = 37, 132
    n = M * N if op == "scale_cols" else 100003
    a = (torch.randn(n, device=DEV, generator=g) * 3).to(at)
    b = (torch.randn(n, device=DEV, generator=g) * 3).to(bt) if bt is not None else None
    gm = torch.randn(N, device=DEV, generator=g)
    bo, out = guarded((n,), ot)

    def call():
        if op == "scale_cols":
            rc = lib().asis_scale_cols(ptr(a), _lib.dt(a), ptr(gm), ptr(out), _lib.dt(out), M, N, _lib.stream())
        elif op == "add":
            rc = lib().asis_add(ptr(a), _lib.dt(a), ptr(b), _lib.dt(b), ptr(out), _lib.dt(out), n, _lib.stream())
        else:
            rc = lib().asis_cast(ptr(a), _lib.dt(a), ptr(out), _lib.dt(out), n, _lib.stream())
        _lib.check(rc)
    run_traced(call, elementwise_plan(op, at, bt, ot, n))
    intact([bo], op)
    if op == "scale_cols":
        ref = (a.float().view(M, N) * gm).reshape(-1).to(ot)
    elif op == "add":
        ref = (a.float() + b.float()).to(ot)
    else:
        ref = a.float().to(ot)
    assert torch.equal(bits(out), bits(ref)), f"{op} differs from torch at {int((bits(out) != bits(ref)).nonzero()[0])}"


# ---------------------------------------------------------------------------------------- depth-wise convolution
PYRAMID = [(73, 73), (36, 36), (18, 18)]
ODD_MAPS = [(7, 5), (1, 9), (9, 1), (1, 1)]
# (name, B, maps, C, fuse, accumulate)
DWCONV_SHAPES = [("vit-l", 12, PYRAMID, 256, True, False), ("vit-b", 12, PYRAMID, 192, True, False),
                 ("odd-fused", 3, ODD_MAPS, 132, True, False), ("odd-unfused", 3, ODD_MAPS, 132, False, True),
                 ("c1280", 2, [(7, 5), (3, 4)], 1280, True, False)]
DWCONV = [(t, s[0]) for t in DTS for s in DWCONV_SHAPES]


def _maps_arrays(maps):
    return (ctypes.c_int * len(maps))(*[h for h, _ in maps]), (ctypes.c_int * len(maps))(*[w for _, w in maps])


def abi_dw_fwd(x, weight, bias, maps, fuse, save_pre):
    B, ntok, C = x.shape
    hs, ws_ = _maps_arrays(maps)
    by, y = guarded((B, ntok, C), x.dtype)
    bp, pre = guarded((B, ntok, C), x.dtype)
    _lib.check(lib().asis_dwconv3x3_forward(ptr(x), _lib.dt(x), ptr(weight), ptr(bias), ptr(pre) if save_pre else None,
                                            ptr(y), B, C, len(maps), hs, ws_, int(fuse), _lib.stream()))
    return y, pre, [by, bp]


def abi_dw_bwd(dy, pre, x, weight, maps, fuse, prior):
    B, ntok, C = x.shape
    hs, ws_ = _maps_arrays(maps)
    bx, dx = guarded((B, ntok, C), x.dtype)
    bw, dw = guarded((C, 9), F32)
    bb, db = guarded((C,), F32)
    if prior is not None:
        dw.copy_(prior[0])
        db.copy_(prior[1])
    nbytes = lib().asis_dwconv3x3_backward_workspace_bytes(B, C, ntok)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    _lib.check(lib().asis_dwconv3x3_backward(ptr(dy), ptr(pre) if fuse else None, ptr(x), _lib.dt(x), ptr(weight),
                                             ptr(dx), ptr(dw), ptr(db), int(prior is not None), B, C, len(maps), hs,
                                             ws_, int(fuse), ptr(ws), nbytes, _lib.stream()))
    return (dx, dw, db), [bx, bw, bb]


@pytest.mark.parametrize("t,name", DWCONV, ids=[f"{TAG[t]}-{n}" for t, n in DWCONV])
def test_dwconv(t, name):
    t0 = time.time()
    _, B, maps, C, fuse, acc = next(s for s in DWCONV_SHAPES if s[0] == name)
    ntok = sum(h * w for h, w in maps)
    g = gen(C + B)
    x = torch.randn(B, ntok, C, device=DEV, generator=g).to(t)
    weight = torch.randn(C, 9, device=DEV, generator=g) * 0.5
    bias = torch.randn(C, device=DEV, generator=g)
    dy = torch.randn(B, ntok, C, device=DEV, generator=g).to(t)
    prior = (torch.randn(C, 9, device=DEV, generator=g), torch.randn(C, device=DEV, generator=g)) if acc else None
    tag = f"dwconv {TAG[t]} {name} B={B} C={C} fuse={fuse}"
    y, pre, bufs = run_traced(lambda: abi_dw_fwd(x, weight, bias, maps, fuse, True), dwconv_fwd_plan(t, B, ntok, C))
    intact(bufs, tag)
    if fuse:                                    # the forward without the saved pre-activation: the same y, pre untouched
        y2, pre2, _ = abi_dw_fwd(x, weight, bias, maps, fuse, False)
        assert torch.equal(bits(y), bits(y2)) and bool((bits(pre2) == R.NAN_BITS[pre2.element_size()]).all())
    else:
        assert bool((bits(pre) == R.NAN_BITS[pre.element_size()]).all()), "unfused forward wrote pre"
    outs, bufs = run_traced(lambda: abi_dw_bwd(dy, pre, x, weight, maps, fuse, prior),
                            dwconv_bwd_plan(t, B, ntok, C, fuse))
    intact(bufs, tag)
    again, _ = abi_dw_bwd(dy, pre, x, weight, maps, fuse, prior)
    assert same_bits(outs, again), f"[{tag}] the backward is not run-to-run identical"
    u = R.u_out(t)
    slabs = NR.dw_slabs(maps)
    rf = NR.dwconv_fwd_ref(x, weight, bias, maps, fuse, t)
    reps = [R.check("y", y, rf["y"][0], u, rf["y"][1], block=slabs)]
    if fuse:
        reps.append(R.check("pre", pre, rf["pre"][0], u, rf["pre"][1], block=slabs))
    del rf
    rb = NR.dwconv_row_blocks(B * ntok, C)
    rr = NR.dwconv_bwd_ref(dy, pre, x, weight, maps, fuse, t, rb, *(prior or (None, None)))
    reps.append(R.check("dx", outs[0], rr["dx"][0], u, rr["dx"][1], block=slabs))
    reps.append(R.check("dweight", outs[1], rr["dweight"][0], R.U_F32, rr["dweight"][1], block=NR.col_slabs))
    reps.append(R.check("dbias", outs[2], rr["dbias"][0], R.U_F32, rr["dbias"][1], block=NR.col_slabs))
    del rr
    report(tag, reps, t0)


# ------------------------------------------------------------------------------------------------- coverage
def every_instantiation():
    """The 61 kernels the launchers of norm.cu and the depth-wise convolution can pick."""
    n = {f"ln_fwd_kernel<{VT[a]},{VT[b]},{nv}>" for a in DTS for b in DTS for nv in NV_CS}
    n |= {f"ln_bwd2_kernel<{VT[a]},{VT[b]}>" for a in DTS for b in DTS}
    n |= {"reduce_partials_kernel<8>", "reduce_partials_kernel<32>"}
    n |= {f"colsum_kernel<{VT[a]},{VT[b]},1>" for a in DTS for b in DTS} | {f"colsum_kernel<{VT[a]},float,0>" for a in DTS}
    n |= {f"layerscale_bwd_kernel<{VT[a]}>" for a in DTS}
    n |= {f"scale_cols_kernel<{VT[a]},{VT[o]}>" for a in DTS for o in DTS}
    n |= {f"add_cast_kernel<{VT[a]},{VT[b]},{VT[o]},1>" for a in DTS for b in DTS for o in DTS}
    n |= {f"add_cast_kernel<{VT[a]},{VT[a]},{VT[o]},0>" for a in DTS for o in DTS}
    for k in ("dwconv_fwd_kernel", "dwconv_bwd_kernel", "dwconv_gelu_grad_kernel"):
        n |= {f"{k}<{VT[a]}>" for a in DTS}
    return n | {"dwconv_reduce_kernel"}


def test_every_instantiation_asserted():
    """The cases above assert, together, every instantiation (each case asserts its plan, so the union of the plans is
    what the file asserts)."""
    plans = []
    for xt, yt, nv in LN_FWD:
        plans += ln_fwd_plan(xt, yt, 7, NV_CS[nv][0])
    for dt, xt, _ in LN_BWD:
        for R_, C, wg, wb, _ in LN_BWD_SHAPES:
            plans += ln_bwd_plan(dt, xt, R_, C, wg, wb)
    for xt, yt in COLSUM:
        for M, N, *_ in COLSUM_SHAPES:
            plans += colsum_plan(xt, yt, M, N)
    for ut, mode in LAYERSCALE:
        plans += layerscale_plan(ut, 21180, 1024, mode != "dbias", mode != "dgamma")
    for op, a, b, o in ELEMENTWISE:
        plans += elementwise_plan(op, a, b, o, 100003)
    for t, name in DWCONV:
        _, B, maps, C, fuse, _ = next(s for s in DWCONV_SHAPES if s[0] == name)
        ntok = sum(h * w for h, w in maps)
        plans += dwconv_fwd_plan(t, B, ntok, C) + dwconv_bwd_plan(t, B, ntok, C, fuse)
    asserted = {p[0] for p in plans}
    want = every_instantiation()
    assert len(want) == 61
    assert not want - asserted, f"instantiations no case asserts: {sorted(want - asserted)}"
    print(f"[coverage] {len(want & asserted)} of {len(want)} instantiations asserted; peak memory "
          f"{torch.cuda.max_memory_allocated() / 2 ** 30:.2f} GB")
