"""The elementwise bounds of tests/norm_ref.py accept what the LayerNorm, column-sum and depth-wise convolution kernels
compute and reject results that are wrong in the ways these kernels go wrong.  No GPU: host models repeat the kernels'
fp32 arithmetic in their order (lane chains, xor butterflies, the 8-warp tree, per-thread column chains over the rows a
block owns, reduce_partials' four accumulators and part-lane chain, the convolution's tap chain at clamped neighbour
indices), with every multiply-add either fused or not, and each mutant breaks one statistic, index or term the way a
bug would."""
import pytest
import torch

import norm_ref as NR
import tc_ref as R

BF, F32 = torch.bfloat16, torch.float32
EPS = 1e-6


def mad(acc, a, b, fused):
    """acc + a b in fp32: fmaf (one rounding) or a rounded product and a rounded sum."""
    if fused:
        return (acc.double() + a.double() * b.double()).float()
    return acc + a * b


def butterfly(s):
    """The xor-shuffle warp sum over the last dimension (32 lanes); every lane ends with the same value."""
    lanes = torch.arange(32)
    for o in (16, 8, 4, 2, 1):
        s = s + s[..., lanes ^ o]
    return s[..., 0]


def reduce_model(parts, prior=None, drop=None):
    """reduce_partials<PL>: part-lane y sums parts y, y + PL, ... into t0..t3 (remainder into t0), then (t0 + t1) +
    (t2 + t3), then a chain over the PL part-lanes; `accumulate` adds the prior value.  `drop`: a part left out."""
    nparts, n = parts.shape
    pl = NR.reduce_pl(nparts)
    z = torch.zeros(n)

    def part(p):
        return z if p == drop else parts[p]
    red = []
    for ty in range(pl):
        t0, t1, t2, t3 = z, z, z, z
        p = ty
        while p + 3 * pl < nparts:
            t0, t1, t2, t3 = t0 + part(p), t1 + part(p + pl), t2 + part(p + 2 * pl), t3 + part(p + 3 * pl)
            p += 4 * pl
        while p < nparts:
            t0 = t0 + part(p)
            p += pl
        red.append((t0 + t1) + (t2 + t3))
    t = z
    for r in red:
        t = t + r
    return t if prior is None else prior + t


def reports(outs, refs, u, blocks):
    return {k: R.check(k, outs[k], refs[k][0], u[k], refs[k][1], block=blocks.get(k)) for k in outs}


def accepts(reps):
    for rep in reps.values():
        assert rep.ok, str(rep)


def rejects(reps, name, slabs=None):
    rep = reps[name]
    assert not rep.ok, f"a wrong {name} passed: {rep}"
    if slabs is not None:
        bad = {tuple(i) for i in (rep.slabs > 1).nonzero().tolist()}
        assert bad == set(slabs), (bad, str(rep))


# ------------------------------------------------------------------------------------- LayerNorm forward
def ln_fwd_model(x, g, b, eps=EPS, fused=True, mut=None):
    """ln_fwd_kernel on fp32 values x [R, C]: (y fp32, mean, rstd)."""
    Rn, C = x.shape
    nv = NR.ln_nv(C)
    X = torch.zeros(Rn, nv * 128)
    X[:, :C] = x
    live = torch.zeros(nv * 128, dtype=torch.bool)
    live[:C] = True
    if mut == "drop_last_vector":
        live[C - 4:C] = False
    X = torch.where(live, X, torch.zeros(()))
    Xv, Lv = X.view(Rn, nv, 32, 4), live.view(nv, 32, 4)
    s = torch.zeros(Rn, 32)
    for j in range(nv):
        s = s + (((Xv[:, j, :, 0] + Xv[:, j, :, 1]) + Xv[:, j, :, 2]) + Xv[:, j, :, 3])
    mu = butterfly(s) / C
    sq = torch.zeros(Rn, 32)
    for j in range(nv):
        for i in range(4):
            v = Xv[:, j, :, i]
            if mut == "one_pass":
                sq = torch.where(Lv[j, :, i], mad(sq, v, v, fused), sq)
            else:
                d = v - mu[:, None]
                sq = torch.where(Lv[j, :, i], mad(sq, d, d, fused), sq)
    ss = butterfly(sq)
    if mut == "one_pass":
        var = ss / C - mu * mu
    elif mut == "unbiased":
        var = ss / (C - 1)
    else:
        var = ss / C
    if mut == "eps_outside":
        rs = 1.0 / (torch.sqrt(var) + eps)
    else:
        rs = torch.rsqrt(var + (1e-5 if mut == "eps_1e-5" else eps))
    gg, bb = (b, g) if mut == "swap_gamma_beta" else (g, b)
    y = mad(bb.expand(Rn, C), (x - mu[:, None]) * rs[:, None], gg.expand(Rn, C), fused)
    return y, mu, rs


def ln_rows(C, seed=0):
    """randn * 2 + 0.5 rows, rows of std 1e-3, rows at a mean offset of 300, a constant and a zero row, an outlier."""
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(24, C, generator=gen) * 2 + 0.5
    x[0:4] = 0.5 + 1e-3 * torch.randn(4, C, generator=gen)
    x[4:8] = 300 + torch.randn(4, C, generator=gen)
    x[8] = 0.7
    x[9] = 0.0
    x[10, 5] = 1e3
    g = torch.randn(C, generator=gen)
    b = torch.randn(C, generator=gen)
    return x, g, b


def ln_fwd_reports(x, g, b, outs, dtype=F32):
    nv = NR.ln_nv(x.shape[1])
    refs = NR.ln_fwd_ref(x, g, b, EPS, nv)
    u = {"y": R.u_out(dtype), "mean": R.U_F32, "rstd": R.U_F32}
    y, mu, rs = outs
    return reports({"y": y.to(dtype), "mean": mu, "rstd": rs}, refs, u,
                   {"y": NR.row_slabs(8), "mean": NR.row_slabs(8), "rstd": NR.row_slabs(8)})


@pytest.mark.parametrize("C", [132, 256, 772])
@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("dtype", [F32, BF])
def test_ln_fwd_model_accepted(C, fused, dtype):
    x, g, b = ln_rows(C)
    if dtype == BF:
        x = x.bfloat16().float()
    accepts(ln_fwd_reports(x, g, b, ln_fwd_model(x, g, b, fused=fused), dtype))


@pytest.mark.parametrize("mut,name", [
    ("unbiased", "rstd"),               # sum of squares over C - 1
    ("eps_outside", "rstd"),            # 1 / (sqrt(var) + eps): seen on the rows of std 1e-3
    ("eps_1e-5", "rstd"),               # nn.LayerNorm's default eps instead of the model's 1e-6
    ("one_pass", "rstd"),               # E[x^2] - E[x]^2 in fp32: cancels at a mean offset of 300
    ("drop_last_vector", "mean"),       # the last 4-vector of a C = 132 row (lane 0, j = 1) left out
    ("swap_gamma_beta", "y"),
])
def test_ln_fwd_mutant_rejected(mut, name):
    x, g, b = ln_rows(132)
    rejects(ln_fwd_reports(x, g, b, ln_fwd_model(x, g, b, mut=mut)), name)


def test_ln_fwd_eps_outside_needs_the_small_rows():
    """eps outside the square root is caught on the rows of std 1e-3 (row block 0) and the constant and zero rows
    (block 1), not on the rows of std 2 (block 2): the cases need rows of small variance."""
    x, g, b = ln_rows(132)
    rejects(ln_fwd_reports(x, g, b, ln_fwd_model(x, g, b, mut="eps_outside")), "rstd", slabs=[(0,), (1,)])


# ------------------------------------------------------------------------------------ LayerNorm backward
def ln_bwd_model(dy, x, g, mu, rs, dres, grid, fused=True, mut=None, prior=None):
    """ln_bwd2_kernel + reduce_partials on fp32 values: (dx, dgamma, dbeta)."""
    Rn, C = x.shape
    xh = (x - mu[:, None]) * rs[:, None]
    t = dy * g
    pad = torch.zeros(Rn, 1024)
    tp, xp = pad.clone(), pad.clone()
    tp[:, :C], xp[:, :C] = t, xh
    tp, xp = tp.view(Rn, 8, 32, 4), xp.view(Rn, 8, 32, 4)
    s1, s2 = torch.zeros(Rn, 8, 32), torch.zeros(Rn, 8, 32)
    for i in range(4):
        s1 = s1 + tp[..., i]
        s2 = mad(s2, tp[..., i], xp[..., i], fused)
    w1, w2 = butterfly(s1), butterfly(s2)

    def tree8(w):
        return ((w[:, 0] + w[:, 1]) + (w[:, 2] + w[:, 3])) + ((w[:, 4] + w[:, 5]) + (w[:, 6] + w[:, 7]))
    inv_c = torch.tensor(1.0) / C
    m1, m2 = (tree8(w1) * inv_c)[:, None], (tree8(w2) * inv_c)[:, None]
    if mut == "drop_m2":
        m2 = torch.zeros_like(m2)
    rr = torch.zeros_like(dy) if dres is None else dres
    if mut == "dres_dropped":
        rr = torch.zeros_like(dy)
    dx = rs[:, None] * (mad(dy * g - m1, -xh, m2.expand_as(xh), fused)) + rr
    if mut == "dres_twice":
        dx = dx + rr
    rows = Rn - 1 if mut == "skip_last_row" else Rn
    if mut == "skip_last_row":
        dx[Rn - 1] = 0.0
    xg = x - mu[:, None] if mut == "dgamma_unnormalised" else xh
    dg, db = torch.zeros(grid, C), torch.zeros(grid, C)
    for b in range(grid):
        for row0 in range(2 * b, rows, 2 * grid):
            for r in range(row0, min(row0 + 2, rows)):
                dg[b] = mad(dg[b], dy[r], xg[r], fused)
                db[b] = db[b] + dy[r]
    drop = 1 if mut == "drop_partial" else None
    pg, pb = (None, None) if (prior is None or mut == "accumulate_ignored") else prior
    return dx, reduce_model(dg, pg, drop), reduce_model(db, pb, drop)


def ln_bwd_case(Rn=95, C=132, seed=1):
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(Rn, C, generator=gen) * 2 + 0.5
    dy = torch.randn(Rn, C, generator=gen)
    dres = torch.randn(Rn, C, generator=gen)
    g = torch.randn(C, generator=gen)
    mu = x.mean(1)
    rs = torch.rsqrt(x.var(1, unbiased=False) + EPS)
    prior = (torch.randn(C, generator=gen), torch.randn(C, generator=gen))
    return dy, x, g, mu, rs, dres, prior


def ln_bwd_reports(case, outs, prior=None):
    dy, x, g, mu, rs, dres, _ = case
    grid = NR.ln_bwd_grid(x.shape[0])
    pg, pb = prior if prior is not None else (None, None)
    refs = NR.ln_bwd_ref(dy, x, g, mu, rs, dres, grid, pg, pb)
    dx, dgm, dbt = outs
    return reports({"dx": dx, "dgamma": dgm, "dbeta": dbt}, refs, {k: R.U_F32 for k in refs},
                   {"dx": NR.row_slabs(2), "dgamma": NR.col_slabs, "dbeta": NR.col_slabs})


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("Rn,C", [(95, 132), (3, 1024), (300, 256)])
def test_ln_bwd_model_accepted(fused, Rn, C):
    case = ln_bwd_case(Rn, C)
    grid = NR.ln_bwd_grid(Rn)
    accepts(ln_bwd_reports(case, ln_bwd_model(*case[:6], grid, fused)))
    accepts(ln_bwd_reports(case, ln_bwd_model(*case[:6], grid, fused, prior=case[6]), prior=case[6]))


@pytest.mark.parametrize("mut,name,accumulate", [
    ("drop_m2", "dx", False),
    ("dres_dropped", "dx", False),
    ("dres_twice", "dx", False),
    ("skip_last_row", "dx", False),          # the last row of an odd R (row 94 of 95)
    ("skip_last_row", "dgamma", False),
    ("dgamma_unnormalised", "dgamma", False),
    ("drop_partial", "dgamma", False),       # block 1's partial left out of the reduction
    ("drop_partial", "dbeta", False),
    ("accumulate_ignored", "dgamma", True),
])
def test_ln_bwd_mutant_rejected(mut, name, accumulate):
    case = ln_bwd_case()
    prior = case[6] if accumulate else None
    outs = ln_bwd_model(*case[:6], NR.ln_bwd_grid(95), mut=mut, prior=prior)
    rejects(ln_bwd_reports(case, outs, prior), name)


def test_ln_bwd_last_row_named():
    case = ln_bwd_case()
    outs = ln_bwd_model(*case[:6], NR.ln_bwd_grid(95), mut="skip_last_row")
    rejects(ln_bwd_reports(case, outs), "dx", slabs=[(47,)])


# ------------------------------------------------------------------------------------------ column sums
def colsum_model(store, off, M, N, ld, Ystore=None, fused=True, mut=None, prior=None):
    """colsum_kernel + reduce_partials on fp32 values: X = rows of `store` (flat, pitch ld) at column offset off."""
    rb = NR.colsum_rb(M, N)
    pitch = N if mut == "pitch_N" else ld
    stride = 8 * rb
    flat = store.reshape(-1)
    yflat = None if (Ystore is None or mut == "ignore_Y") else Ystore.reshape(-1)
    acc = torch.zeros(stride, N)
    for t in range(stride):
        rows = list(range(t, M, stride))
        if mut == "drop_remainder":
            rows = rows[:len(rows) // 4 * 4]
        for r in rows:
            a = flat[off + r * pitch:off + r * pitch + N]
            acc[t] = acc[t] + a if yflat is None else mad(acc[t], a, yflat[off + r * pitch:off + r * pitch + N], fused)
    parts = torch.zeros(rb, N)
    for by in range(rb):
        for ty in range(8):
            parts[by] = parts[by] + acc[by * 8 + ty]
    return reduce_model(parts, prior)


def colsum_case(M=1001, N=132, ld=148, off=8, seed=2):
    gen = torch.Generator().manual_seed(seed)
    X = torch.randn(M, ld, generator=gen) + 0.25
    Y = torch.randn(M, ld, generator=gen)
    return X, Y, torch.randn(N, generator=gen)


def colsum_report(X, Y, off, N, out, prior=None):
    ref = NR.colsum_ref(X[:, off:off + N], None if Y is None else Y[:, off:off + N], prior=prior)
    return {"colsum": R.check("colsum", out, ref[0], R.U_F32, ref[1], block=NR.col_slabs)}


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("with_y", [False, True])
@pytest.mark.parametrize("M,N,ld", [(1001, 132, 148), (37, 4, 4), (3000, 64, 64)])
def test_colsum_model_accepted(fused, with_y, M, N, ld):
    X, Y, prior = colsum_case(M, N, ld, 0 if ld == N else 8)
    off = 0 if ld == N else 8
    Ys = Y if with_y else None
    accepts(colsum_report(X, Ys, off, N, colsum_model(X, off, M, N, ld, Ys, fused)))
    accepts(colsum_report(X, Ys, off, N, colsum_model(X, off, M, N, ld, Ys, fused, prior=prior), prior))


@pytest.mark.parametrize("mut", ["drop_remainder", "pitch_N", "ignore_Y"])
def test_colsum_mutant_rejected(mut):
    X, Y, _ = colsum_case()
    rejects(colsum_report(X, Y, 8, 132, colsum_model(X, 8, 1001, 132, 148, Y, mut=mut)), "colsum")


# ---------------------------------------------------------------------------------- depth-wise convolution
DW_MAPS = [(5, 7), (3, 4)]
DW_B, DW_C = 2, 8


def nbr_table(maps, mut=None):
    """[ntok, 9] neighbour token index (clamped coordinates, as the kernels load them) and [ntok, 9] tap-inside mask."""
    ntok = sum(h * w for h, w in maps)
    idx = torch.zeros(ntok, 9, dtype=torch.long)
    ok = torch.zeros(ntok, 9, dtype=torch.bool)
    t0 = 0
    for H, W in maps:
        for p in range(H * W):
            py, px = divmod(p, W)
            for j, (oy, ox) in enumerate(NR.TAPS):
                yy, xx = py + oy, px + ox
                inside = 0 <= yy < H and 0 <= xx < W
                i = t0 + min(max(yy, 0), H - 1) * W + min(max(xx, 0), W - 1)
                if mut == "clamped_tap":
                    inside = True
                elif mut == "token_wrap":                 # horizontal neighbour = token index +- 1
                    i = t0 + yy * W + px + ox
                    inside = 0 <= yy < H and t0 <= i < t0 + H * W
                elif mut == "adjacent_map":               # vertical neighbour by W tokens, past the map's end
                    i = t0 + p + oy * W + ox
                    inside = 0 <= xx < W and 0 <= i < ntok
                idx[t0 + p, j] = i if inside else min(max(i, 0), ntok - 1)
                ok[t0 + p, j] = inside
        t0 += H * W
    return idx, ok


def gelu32(x):
    return 0.5 * x * (1.0 + torch.erf(x * 0.70710678118654752))


def dgelu32(x):
    cdf = 0.5 * (1.0 + torch.erf(x * 0.70710678118654752))
    return cdf + x * (0.3989422804014327 * torch.exp(-0.5 * x * x))


def taps(weight, mut):
    w = weight.reshape(-1, 9)
    if mut == "flipped_taps":
        w = w[:, list(range(8, -1, -1))]
    if mut == "channels_shifted":
        w = w[(torch.arange(w.shape[0]) + 4) % w.shape[0]]
    return w


def dw_fwd_model(x, weight, bias, maps, fuse, dtype, fused=True, mut=None):
    idx, ok = nbr_table(maps, mut)
    w = taps(weight, mut)
    acc = bias.expand(x.shape).clone()
    for j in range(9):
        acc = torch.where(ok[None, :, j, None], mad(acc, x[:, idx[:, j]], w[:, j], fused), acc)
    y = gelu32(acc) if fuse else acc
    return acc.to(dtype), y.to(dtype)


def dw_bwd_model(dy, pre, y, x, weight, maps, fuse, dtype, fused=True, mut=None):
    B, ntok, C = x.shape
    idx, ok = nbr_table(maps, mut)
    w = taps(weight, mut)
    if fuse:
        at = y if mut == "dgelu_at_y" else pre
        g = (dy.float() * dgelu32(at.float())).to(dtype).float()
    else:
        g = dy.float()
    dx = torch.zeros(B, ntok, C)
    for j in range(9):
        dx = torch.where(ok[None, :, 8 - j, None], mad(dx, g[:, idx[:, 8 - j]], w[:, j], fused), dx)
    rows = B * ntok
    rb = NR.dwconv_row_blocks(rows, C)
    gr, xr = g.reshape(rows, C), x.reshape(B * ntok, C)
    skip = set(range(DW_MAPS[0][0] * DW_MAPS[0][1], ntok)) if mut == "drop_map_dbias" else set()
    acc = torch.zeros(8 * rb, 10, C)
    for t in range(8 * rb):
        for r in range(t, rows, 8 * rb):
            b, tok = divmod(r, ntok)
            for j in range(9):
                if ok[tok, j]:
                    acc[t, j] = mad(acc[t, j], gr[r], xr[b * ntok + idx[tok, j]], fused)
            if tok not in skip:
                acc[t, 9] = acc[t, 9] + gr[r]
    parts = torch.zeros(rb, 10, C)
    for by in range(rb):
        for ty in range(8):
            parts[by] = parts[by] + acc[by * 8 + ty]
    tot = torch.zeros(10, C)
    for p in range(rb):
        tot = tot + parts[p]
    return dx.to(dtype), tot[:9].t().contiguous(), tot[9]


def dw_case(dtype, seed=3):
    gen = torch.Generator().manual_seed(seed)
    ntok = sum(h * w for h, w in DW_MAPS)
    x = torch.randn(DW_B, ntok, DW_C, generator=gen)
    s = 0
    for m, (h, w) in enumerate(DW_MAPS):                 # each (image, map) its own offset
        x[:, s:s + h * w] += torch.tensor([1.0, -2.0]).view(DW_B, 1, 1) * (m + 1)
        s += h * w
    weight = torch.randn(DW_C, 1, 3, 3, generator=gen)
    bias = torch.randn(DW_C, generator=gen)
    dy = torch.randn(DW_B, ntok, DW_C, generator=gen).to(dtype).float()
    return x.to(dtype).float(), weight, bias, dy


def dw_reports(dtype, fuse, fwd=None, bwd=None, seed=3):
    x, weight, bias, dy = dw_case(dtype, seed)
    u = {"pre": R.u_out(dtype), "y": R.u_out(dtype), "dx": R.u_out(dtype), "dweight": R.U_F32, "dbias": R.U_F32}
    blocks = {"pre": NR.dw_slabs(DW_MAPS), "y": NR.dw_slabs(DW_MAPS), "dx": NR.dw_slabs(DW_MAPS),
              "dweight": NR.col_slabs, "dbias": NR.col_slabs}
    reps = {}
    pre, y = fwd or dw_fwd_model(x, weight, bias, DW_MAPS, fuse, dtype)
    rf = NR.dwconv_fwd_ref(x, weight, bias, DW_MAPS, fuse, dtype)
    reps.update(reports({"pre": pre, "y": y}, rf, u, blocks))
    if bwd is not None:
        rb = NR.dwconv_row_blocks(x.shape[0] * x.shape[1], DW_C)
        rr = NR.dwconv_bwd_ref(dy, pre.float(), x, weight, DW_MAPS, fuse, dtype, rb)
        dx, dw, db = bwd(x, weight, dy, pre, y)
        reps.update(reports({"dx": dx, "dweight": dw, "dbias": db}, rr, u, blocks))
    return reps


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("fuse", [True, False])
@pytest.mark.parametrize("dtype", [F32, BF])
def test_dwconv_model_accepted(fused, fuse, dtype):
    x, weight, bias, _ = dw_case(dtype)
    fwd = dw_fwd_model(x, weight, bias, DW_MAPS, fuse, dtype, fused)
    accepts(dw_reports(dtype, fuse, fwd, lambda x, w, dy, pre, y: dw_bwd_model(dy, pre, y, x, w, DW_MAPS, fuse, dtype,
                                                                               fused)))


@pytest.mark.parametrize("dtype", [F32, BF])
@pytest.mark.parametrize("mut,name", [
    ("flipped_taps", "y"),              # w[8 - j]
    ("clamped_tap", "y"),               # an outside tap counted with its clamped neighbour's value
    ("token_wrap", "y"),                # the horizontal neighbour by token index +- 1: wraps across rows
    ("adjacent_map", "y"),              # the vertical neighbour read past the map's end, in the adjacent map
    ("channels_shifted", "y"),          # channel c convolved with channel c + 4's taps
    ("flipped_taps", "dx"),
    ("clamped_tap", "dx"),
    ("token_wrap", "dweight"),
    ("adjacent_map", "dweight"),
    ("dgelu_at_y", "dx"),               # GELU' evaluated at y instead of pre
    ("dgelu_at_y", "dbias"),
    ("drop_map_dbias", "dbias"),        # the second map's tokens missing from dbias
])
def test_dwconv_mutant_rejected(dtype, mut, name):
    x, weight, bias, _ = dw_case(dtype)
    fwd_mut = mut if name == "y" else None
    fwd = dw_fwd_model(x, weight, bias, DW_MAPS, True, dtype, mut=fwd_mut)
    bwd = None if name == "y" else \
        (lambda x, w, dy, pre, y: dw_bwd_model(dy, pre, y, x, w, DW_MAPS, True, dtype, mut=mut))
    rejects(dw_reports(dtype, True, fwd, bwd), name)


def test_dwconv_border_slabs_named():
    """A counted outside tap fails in every (image, map) slab (every map has a border) and in no other way."""
    x, weight, bias, _ = dw_case(F32)
    fwd = dw_fwd_model(x, weight, bias, DW_MAPS, True, F32, mut="clamped_tap")
    reps = dw_reports(F32, True, fwd)
    rejects(reps, "y", slabs=[(b, m, 0) for b in range(DW_B) for m in range(len(DW_MAPS))])
