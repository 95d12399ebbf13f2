"""The elementwise bounds of tests/msda_ref.py accept what the deformable-attention kernels compute and reject results
that are wrong in the ways a gather / scatter kernel goes wrong.  No GPU: a host model of the kernels' arithmetic (fp32
corner weights, fp32 fmaf chains in the kernels' order, the locaw lanes' 16-channel chains and shuffle tree, bf16
stores) produces the correct result at a small shape, and each test then breaks one index, mask, weight or row the
way a bug would.  Operands carry an offset and a scale per (image, head, level), so each wrong result is off by O(1)
in its own slab."""
import pytest
import torch

import msda_ref as MR

BF, F32 = torch.bfloat16, torch.float32
N, M, D, P, LQ, QCHUNK = 2, 3, 32, 2, 40, 16
SHAPES = [(5, 7), (3, 4)]            # non-square levels
L = len(SHAPES)
STARTS = MR.level_starts(SHAPES)
S = sum(h * w for h, w in SHAPES)


def fma(acc, a, b):
    """fmaf: the exact product plus acc, rounded once to fp32."""
    return (acc.double() + a.double() * b.double()).float()


def case(dtype, seed=0):
    g = torch.Generator().manual_seed(seed)
    value, gout = MR.operands(g, N, LQ, M, D, SHAPES, dtype)
    loc = MR.sample_locations(g, N, LQ, M, SHAPES, P)
    aw = MR.attention_weights(g, N, LQ, M, L, P)
    return dict(value=value, gout=gout, loc=loc, aw=aw, dtype=dtype)


# ------------------------------------------------------------------------------------------ host model
def points(loc, mut):
    """Per-level footprints as the kernels build them (fp32), with the geometry mutants."""
    pix, mask, cmask, fxs, fys = [], [], [], [], []
    for l, (H, W) in enumerate(SHAPES):
        h, w = (W, H) if (mut == "xy_swap" and l == 0) else (H, W)
        x, y, x0, y0, fx, fy, any_ = MR.footprint(loc[..., l, :, 0], loc[..., l, :, 1], h, w)
        if mut == "left_strip":                     # a point in (-1, 0) taken as outside
            any_ = any_ & (x >= 0)
            x0, fx = torch.where(any_, x0, 0), torch.where(any_, fx, 0.0)
            y0, fy = torch.where(any_, y0, 0), torch.where(any_, fy, 0.0)
        xl, yt, yb = any_ & (x0 >= 0), y0 >= 0, y0 + 1 < h
        xr = any_ & (x0 + 1 <= w) if mut == "right_edge" else any_ & (x0 + 1 < w)
        xa, xb, ya, yc = x0.clamp_min(0), (x0 + 1).clamp_max(w - 1), y0.clamp_min(0), (y0 + 1).clamp_max(h - 1)
        s = STARTS[1] if (mut == "next_start" and l == 0) else STARTS[l]
        p4 = torch.stack([s + ya * w + xa, s + ya * w + xb, s + yc * w + xa, s + yc * w + xb], -1).clamp_max(S - 1)
        m4 = torch.stack([yt & xl, yt & xr, yb & xl, yb & xr], -1)
        pix.append(p4)
        mask.append(m4)
        cmask.append(any_[..., None].expand_as(m4) if mut == "ga_clamped" else m4)
        fxs.append(fx)
        fys.append(fy)
    return (torch.stack(pix, -3), torch.stack(mask, -3), torch.stack(cmask, -3), torch.stack(fxs, -2),
            torch.stack(fys, -2))


def model(c, mut=None, entry=None):
    """out, grad_value, grad_loc, grad_attn as the kernels compute them."""
    value, loc, aw, dtype = c["value"], c["loc"], c["aw"].clone(), c["dtype"]
    if mut == "neighbour_aw":
        aw = aw[..., torch.arange(P) ^ 1]
    v = value.float()
    if mut == "head_slice":                          # (image 1, head 0) reads head 1's value slice
        v = v.clone()
        v[1, :, 0] = v[1, :, 1]
    go = c["gout"].float().view(N, LQ, M, D)
    pix, mask, cmask, fx, fy = points(loc, mut)
    nn = torch.arange(N).view(N, 1, 1, 1, 1, 1)
    mm = torch.arange(M).view(1, 1, M, 1, 1, 1)
    vc = v[nn, pix, mm]                                                          # [N, Lq, M, L, P, 4, D]
    ofx, ofy = 1.0 - fx, 1.0 - fy
    a = aw
    m = mask.float()
    w01x = ofx if mut == "swap_fx" else fx
    w = torch.stack([ofx * ofy * a, w01x * ofy * a, ofx * fy * a, fx * fy * a], -1) * m
    # forward: one fmaf chain over (level, point, corner)
    acc = torch.zeros(N, LQ, M, D)
    for l in range(L):
        for p in range(P):
            for k in range(4):
                acc = fma(acc, w[:, :, :, l, p, k, None], vc[:, :, :, l, p, k])
    out = acc.to(dtype)
    # locaw: lanes of 16 channels (vector g + GP k), fmaf chains, lane combination, shuffle tree
    cpl = 8 if dtype == BF and D % 8 == 0 else 4
    gp, nv = MR.locaw_gp(D), D // cpl
    lanes = []
    for g in range(gp):
        chans = [cpl * vi + i for vi in range(g, nv, gp) for i in range(cpl)]
        t = torch.zeros(N, LQ, M, L, P, 4)
        for ch in chans:
            t = fma(t, go[:, :, :, None, None, None, ch], vc[..., ch])
        t = t * cmask.float()
        t00, t01, t10, t11 = t.unbind(-1)
        top, bot = ofx * t00 + fx * t01, ofx * t10 + fx * t11
        lanes.append((ofy * top + fy * bot, ofy * (t01 - t00) + fy * (t11 - t10), bot - top))
    step = gp // 2
    while step:                                      # __shfl_xor tree: lane i + lane i ^ step
        lanes = [tuple(x + y for x, y in zip(lanes[i], lanes[i ^ step])) for i in range(len(lanes))]
        step //= 2
    d_a, d_x, d_y = lanes[0]
    Wf = torch.tensor([float(wd) for _, wd in SHAPES]).view(L, 1)
    Hf = torch.tensor([float(ht) for ht, _ in SHAPES]).view(L, 1)
    gl = torch.stack([(a * (Hf if mut == "gl_scale_H" else Wf)) * d_x, (a * Hf) * d_y], -1)
    # grad_value: every pixel's entries in query order, one fmaf chain per pixel
    wf = torch.stack([ofx * ofy * a, fx * ofy * a, ofx * fy * a, fx * fy * a], -1)
    gv = torch.zeros(N, S, M, D)
    n2, m2 = torch.arange(N).view(N, 1), torch.arange(M).view(1, M)
    for q in range(LQ):
        qs = q - 1 if (mut == "prev_row" and q % QCHUNK == 0 and q > 0) else q
        for l in range(L):
            for p in range(P):
                for k in range(4):
                    pk, mk = pix[:, q, :, l, p, k], mask[:, q, :, l, p, k].clone()
                    reps = 1
                    if entry is not None and (q, l, p, k) == entry[2:]:
                        sel = (n2 == entry[0]) & (m2 == entry[1])
                        if mut == "drop_entry":
                            mk &= ~sel
                        else:
                            reps = 2
                    for r in range(reps):
                        if r == 1:
                            mk = mk & sel
                        cur = gv[n2, pk, m2]
                        new = fma(cur, wf[:, q, :, l, p, k, None], go[:, qs])
                        gv[n2, pk, m2] = torch.where(mk[..., None], new, cur)
    return dict(out=out, grad_value=gv.to(dtype), grad_loc=gl, grad_attn=d_a)


def prep_model(off, logits, ref, mut=None):
    """loc, attn of the prep forward (fp32, sequential row sums) for 2-wide reference points with one row per query."""
    lg = logits.float().view(N, LQ, M, L * P)
    if mut == "softmax_head":
        lg = lg[:, :, (torch.arange(M) + 1) % M]
    mx = lg.amax(-1, keepdim=True)
    s = torch.zeros(N, LQ, M, 1)
    for i in range(L * P):
        s = s + torch.exp(lg[..., i:i + 1] - mx)
    attn = torch.exp(lg - mx) * (1.0 / s)
    wh = torch.tensor([[float(w), float(h)] for h, w in SHAPES]).view(L, 1, 2)
    rp = ref.float().view(1, LQ, 1, 1, 1, 2)
    loc = rp + off.float().view(N, LQ, M, L, P, 2) / wh
    return loc, attn.view(N, LQ, M, L, P)


def prep_bwd_model(gloc, gattn, attn, out_dtype):
    a, g = attn.view(N, LQ, M, L * P), gattn.view(N, LQ, M, L * P)
    dot = torch.zeros(N, LQ, M, 1)
    for i in range(L * P):
        dot = fma(dot, g[..., i:i + 1], a[..., i:i + 1])
    wh = torch.tensor([[float(w), float(h)] for h, w in SHAPES]).view(L, 1, 2)
    return (gloc.view(N, LQ, M, L, P, 2) / wh).to(out_dtype), (a * (g - dot)).to(out_dtype).view(N, LQ, M, L, P)


# --------------------------------------------------------------------------------------------- helpers
_REFS = {}


def refs(dtype):
    if dtype not in _REFS:
        c = case(dtype)
        _REFS[dtype] = (c, MR.msda_refs(c["value"], SHAPES, c["loc"], c["aw"], c["gout"]))
    return _REFS[dtype]


def reports(c, r, outs):
    return {rep.name: rep for rep in MR.check_all(outs, r, c["dtype"], SHAPES)}


def accepts(reps):
    for rep in reps.values():
        assert rep.ok, str(rep)


def rejects(reps, name, slabs=None):
    """`name` fails its bound; with `slabs`, exactly those slabs fail."""
    rep = reps[name]
    assert not rep.ok, f"a wrong {name} passed: {rep}"
    if slabs is not None:
        bad = {tuple(i) for i in (rep.slabs > 1).nonzero().tolist()}
        assert bad == set(slabs), (bad, str(rep))


# ----------------------------------------------------------------------------------------------- tests
def test_placements_are_exact():
    """The sample generator puts pixel coordinates exactly on borders, on -1 and on the size, and inside the two
    one-column strips, as the kernel computes them."""
    c = case(F32)
    for l, (H, W) in enumerate(SHAPES):
        for ax, n in ((0, W), (1, H)):
            x = MR._pix(c["loc"][..., l, :, ax], n)
            assert (x == n).any() and (x == n - 1).any()
            assert (x == -1).any() or n & (n - 1) != 0       # reachable exactly for power-of-two sizes only
            assert ((x > -1) & (x < 0)).any() and ((x > n - 1) & (x < n)).any()
            assert ((x == torch.floor(x)) & (x > 0) & (x < n - 1)).any()
            assert ((x < -2) | (x > n + 1)).any()


@pytest.mark.parametrize("dtype", [F32, BF])
def test_model_accepted(dtype):
    c, r = refs(dtype)
    reps = reports(c, r, model(c))
    accepts(reps)
    # pixels no in-map corner touches have a zero reference and a zero bound
    assert (r["grad_value"][1][0][1] == 0).any()


@pytest.mark.parametrize("dtype", [F32, BF])
@pytest.mark.parametrize("mut,name", [
    ("swap_fx", "out"),                 # fx and 1 - fx exchanged on corner 01
    ("xy_swap", "out"),                 # x / y sizes exchanged on the 5 x 7 level
    ("next_start", "out"),              # level 0 read at level 1's start
    ("right_edge", "out"),              # a corner at x0 + 1 = W counted: the clamped pixel with weight fx
    ("left_strip", "out"),              # a point with x in (-1, 0) dropped as outside
    ("neighbour_aw", "out"),            # the neighbouring point's attention weight
    ("prev_row", "grad_value"),         # the previous query's grad_out row for the first query of a chunk
    ("gl_scale_H", "grad_loc"),         # grad_loc x scaled by H
    ("ga_clamped", "grad_attn"),        # an outside corner's clamped value counted in grad_attn
])
def test_mutant_rejected(dtype, mut, name):
    c, r = refs(dtype)
    rejects(reports(c, r, model(c, mut)), name)


@pytest.mark.parametrize("dtype", [F32, BF])
def test_head_slice_named(dtype):
    """(image 1, head 0) reading head 1's value slice fails in exactly that slab."""
    c, r = refs(dtype)
    reps = reports(c, r, model(c, "head_slice"))
    rejects(reps, "out", slabs=[(1, 0)])
    rejects(reps, "grad_attn", slabs=[(1, 0)])


def _heaviest_entry(c, n, m):
    """(n, m, q, l, p, corner) of the in-map grad_value entry with the largest weight in (image n, head m)."""
    geo = MR.geometry(c["loc"], SHAPES)
    bil, _, _ = MR._bilinear(geo["fx"], geo["fy"], geo["mask"])
    w = bil[n, :, m] * c["aw"][n, :, m, :, :, None].double()
    q, l, p, k = torch.unravel_index(w.argmax(), w.shape)
    return (n, m, int(q), int(l), int(p), int(k))


@pytest.mark.parametrize("dtype", [F32, BF])
@pytest.mark.parametrize("mut", ["drop_entry", "dup_entry"])
def test_grad_value_entry_named(dtype, mut):
    """One grad_value entry dropped, or one duplicated, fails in exactly its (image, level, head) slab."""
    c, r = refs(dtype)
    e = _heaviest_entry(c, 1, 2)
    rejects(reports(c, r, model(c, mut, entry=e)), "grad_value", slabs=[(1, e[3], 2)])


def _prep_case(dtype, ref_dim):
    g = torch.Generator().manual_seed(3)
    off = (torch.randn(N, LQ, M * L * P * 2, generator=g) * 2).to(dtype)
    logits = (torch.randn(N, LQ, M * L * P, generator=g) * 3).to(dtype)
    ref = torch.rand(1, LQ, 1, ref_dim, generator=g)
    return off, logits, ref


@pytest.mark.parametrize("dtype", [F32, BF])
def test_prep_model_accepted_softmax_head_rejected(dtype):
    off, logits, ref = _prep_case(dtype, 2)
    r = MR.prep_forward_refs(off, logits, ref, SHAPES, N, LQ, M, L, P)
    import tc_ref as R

    def reps(loc, attn):
        return {k: R.check(k, o, r[k][0], R.U_F32, r[k][1], block=MR.query_slabs)
                for k, o in (("loc", loc), ("attn", attn))}
    accepts(reps(*prep_model(off, logits, ref)))
    rejects(reps(*prep_model(off, logits, ref, "softmax_head")), "attn")
    # backward: grad_offsets, grad_logits
    g = torch.Generator().manual_seed(4)
    gloc, gattn = torch.randn(N, LQ, M, L, P, 2, generator=g), torch.randn(N, LQ, M, L, P, generator=g)
    _, attn = prep_model(off, logits, ref)
    rb = MR.prep_backward_refs(gloc, gattn, attn, ref, SHAPES, dtype, N, LQ, M, L, P)
    goff, glog = prep_bwd_model(gloc, gattn, attn, dtype)
    for k, o in (("grad_offsets", goff), ("grad_logits", glog)):
        rep = R.check(k, o, rb[k][0], R.u_out(dtype), rb[k][1], block=MR.query_slabs)
        assert rep.ok, str(rep)
