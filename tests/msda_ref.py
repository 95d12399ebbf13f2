"""fp64 references with elementwise error bounds for the multi-scale deformable attention kernels (csrc/msda.cu): the
forward, the backward's grad_value / grad_loc / grad_attn, and the softmax / sampling-location prep with its backward.

The rule is tc_ref's (its `check` is used as is): a kernel result passes when, element by element,

    |kernel - ref|  <=  u_out |ref|  +  sum_k c_k shadow_k

with u_out the unit roundoff of the stored type (2^-8 bf16, 2^-24 f32) and each shadow the same expression evaluated on
absolute values.  A rounding of a value that is already off by e adds (1 + u_out) e; the constants carry that factor.

Exact footprint.  The kernels choose a sample's bilinear cell by floor() of its pixel coordinate
x = ((2 lx - 1 + 1) W - 1) / 2, evaluated in fp32 with one explicit round-to-nearest per step (__fmul_rn / __fadd_rn).
`footprint` repeats those steps one fp32 torch op at a time, so it reproduces the kernel's x, floor(x), fx = x - floor(x)
(exact in fp32) and the in-map test bit for bit.  Everything after that is evaluated in fp64 on what the kernel reads:
the value in its own dtype and grad_out cast to the value dtype (as kernels.msda_backward does).  Because the reference
uses the kernel's own cell, samples may sit exactly on integer coordinates and on the map's border: the derivative's
jump there is not an ambiguity.

Constants.  gamma(n) = n u / (1 - n u), u = 2^-24, bounds the relative error of n successive fp32 roundings of
products and sums of non-negative weights (Higham, Accuracy and Stability of Numerical Algorithms, Lemma 3.1 / 3.4);
gamma(a) + gamma(b) <= gamma(a + b).  Products of bf16 or f32 operands are rounded once by fmaf.
  * corner weight w_c = (1 - fx)(1 - fy) a (and its three siblings): 1 - fx, 1 - fy, two products -> gamma(4)
    (the fill kernel forms the same four roundings for grad_value's entries).
  * forward, one fmaf chain of 4 L P corners per channel: gamma(4 L P) on top of the weights -> c = gamma(4 L P + 4),
    shadow sum_c |w_c| |v_c|.
  * locaw (grad_attn, grad_loc): each lane forms t_c = <grad_out, v_c> over its 16 channels by fmaf (gamma(16) of
    sum |go||v_c|); the lane's combination of the four t_c has at most six roundings on any path (1 - fx, 1 - fy, two
    products, two sums for d_attn; the difference, 1 - fy, product and sum for d_x; two products and two sums for
    d_y); the shuffle tree adds log2(GP) sums, and d_loc takes two more products (a W, then times d_x) ->
    c = gamma(22 + log2 GP) for both outputs.  Shadows: grad_attn sum_c bil_c T_c;
    grad_loc x a W (ofy (T00 + T01) + fy (T10 + T11)), y a H (ofx (T00 + T10) + fx (T01 + T11)) (d_y = bot - top
    cancels, the shadow does not), with T_c = sum_ch |go| |v_c| of the corners inside the map.
  * gather (grad_value): the pixel's entries are summed by one fmaf chain whose length is the pixel's entry count k,
    on weights with four roundings -> c = gamma(k + 4), a tensor: k is counted per (image, head, pixel) here.
    Shadow sum_entries |w| |go|.  A pixel that no in-map corner touches has bound 0: it must be exactly 0.
  * prep forward: d_i = lg_i - max is rounded once (a relative error of u |d_i| of exp(d_i)) and expf is within
    2 ulp (2^-22 relative), so each exponential errs by delta_i = 2^-24 |d_i| + 2^-22; the fp32 row sum adds
    gamma(LP - 1) and the max of delta, 1 / sum and the product one rounding each ->
    attn: c = (delta_i + max_j delta_j + gamma(LP + 1))(1 + 2^-20), shadow attn (the factor covers the second-order
    products of these terms, < 2^-30 of them at LP <= 64 and |d| < 2^8).  Below 2^-126 relative bounds fail: an
    exponential or a weight in the subnormal range errs by up to 2 ulp of 2^-149, and the product by half of one,
    hence an absolute 2^-147.
    loc = ref + off / W: the division and the sum (the stored value) -> c = 2 u of |off / W|; with 4-wide reference
    points ref + off / P * w * 0.5: division and product -> gamma(2)(1 + u) of |off w / (2 P)|.
  * prep backward: dot = sum_j ga_j a_j sequentially (gamma(LP) of sum |ga| a), ga_i - dot and the product one
    rounding each -> grad_logits c = gamma(LP + 2)(1 + u_out), shadow a (|ga| + sum_j |ga_j| a_j), plus the
    subnormal rounding of the product and of the store (2^-150 + half the output's smallest subnormal spacing);
    grad_offsets = gloc / W (one rounding; 4-wide points: / P, * w, two) -> c = gamma(1 or 2)(1 + u_out) of |ref|.

Slabs: query-side outputs report the worst ratio per (image, head), grad_value per (image, level, head), so a unit that
read another unit's data is named.
"""
import math

import torch

import tc_ref as R

U = R.U_F32


def gamma(n):
    return n * U / (1.0 - n * U)


def group_pad(g):
    gp = 1
    while gp < g:
        gp <<= 1
    return gp


def locaw_gp(D):
    """Lanes per (query, head) of the backward's locaw kernel: 16 channels per lane, padded to a power of two."""
    return group_pad((D + 15) // 16)


def level_starts(shapes):
    st, s = [], 0
    for h, w in shapes:
        st.append(s)
        s += h * w
    return st


# -------------------------------------------------------------------------------------------- footprint
def _pix(t, n):
    """The kernel's pixel coordinate ((2 t - 1 + 1) n - 1) / 2, one fp32 rounding per step."""
    t = t.float() * 2.0
    t = t + (-1.0)
    t = t + 1.0
    t = t * float(n)
    t = t + (-1.0)
    return t * 0.5


def footprint(lx, ly, H, W):
    """footprint() of csrc/msda.cu on fp32 tensors: (x, y, x0, y0, fx, fy, any), x0 / y0 long, fx / fy fp32."""
    x, y = _pix(lx, W), _pix(ly, H)
    any_ = (x > -1.0) & (x < float(W)) & (y > -1.0) & (y < float(H))
    xf, yf = torch.floor(x), torch.floor(y)
    zero = torch.zeros_like(x)
    x0 = torch.where(any_, xf, zero).long()
    y0 = torch.where(any_, yf, zero).long()
    fx = torch.where(any_, x - xf, zero)
    fy = torch.where(any_, y - yf, zero)
    return x, y, x0, y0, fx, fy, any_


def geometry(loc, shapes):
    """loc [..., L, P, 2] f32 -> dict of pix [..., L, P, 4] (the clamped pixel index into S of corners 00, 01, 10, 11),
    mask [..., L, P, 4] (corner inside the map), fx, fy [..., L, P] (fp32 fractions, 0 outside), W, H [L, 1]."""
    starts = level_starts(shapes)
    pix, mask, fxs, fys = [], [], [], []
    for l, (H, W) in enumerate(shapes):
        _, _, x0, y0, fx, fy, any_ = footprint(loc[..., l, :, 0], loc[..., l, :, 1], H, W)
        xl, xr = any_ & (x0 >= 0), any_ & (x0 + 1 < W)
        yt, yb = y0 >= 0, y0 + 1 < H
        xa, xb = x0.clamp_min(0), (x0 + 1).clamp_max(W - 1)
        ya, yc = y0.clamp_min(0), (y0 + 1).clamp_max(H - 1)
        s = starts[l]
        pix.append(torch.stack([s + ya * W + xa, s + ya * W + xb, s + yc * W + xa, s + yc * W + xb], -1))
        mask.append(torch.stack([yt & xl, yt & xr, yb & xl, yb & xr], -1))
        fxs.append(fx)
        fys.append(fy)
    dev = loc.device
    return dict(pix=torch.stack(pix, -3), mask=torch.stack(mask, -3), fx=torch.stack(fxs, -2),
                fy=torch.stack(fys, -2),
                W=torch.tensor([float(w) for _, w in shapes], dtype=torch.float64, device=dev)[:, None],
                H=torch.tensor([float(h) for h, _ in shapes], dtype=torch.float64, device=dev)[:, None])


def _bilinear(fx, fy, mask):
    """fp64 corner weights, their d / d x and d / d y (pixel units), all zero on corners outside the map."""
    fx, fy = fx.double(), fy.double()
    ox, oy = 1.0 - fx, 1.0 - fy
    m = mask.double()
    bil = torch.stack([ox * oy, fx * oy, ox * fy, fx * fy], -1) * m
    dbx = torch.stack([-oy, oy, -fy, fy], -1) * m
    dby = torch.stack([-ox, -fx, ox, fx], -1) * m
    return bil, dbx, dby


# ------------------------------------------------------------------------------------------- references
def msda_refs(value, shapes, loc, aw, gout=None):
    """References of the forward (and, with gout [N, Lq, M*D], of the backward) in fp64, evaluated one (image, head)
    at a time on value's device.  Returns {name: (ref, terms)}:
      out [N, Lq, M, D], grad_value [N, S, M, D], grad_loc [N, Lq, M, L, P, 2], grad_attn [N, Lq, M, L, P]."""
    N, S, M, D = value.shape
    _, Lq, _, L, P, _ = loc.shape
    dev = value.device
    geo = geometry(loc.to(dev).float(), shapes)
    bil, dbx, dby = _bilinear(geo["fx"], geo["fy"], geo["mask"])
    a = aw.to(dev).double()
    K4 = L * P * 4
    f64 = dict(dtype=torch.float64, device=dev)
    out, out_sh = torch.empty(N, Lq, M, D, **f64), torch.empty(N, Lq, M, D, **f64)
    refs = {}
    if gout is not None:
        go_all = gout.to(dev).to(value.dtype).view(N, Lq, M, D)
        gv, gv_sh, gv_c = (torch.zeros(N, S, M, D, **f64), torch.zeros(N, S, M, D, **f64),
                           torch.empty(N, S, M, 1, **f64))
        gl, gl_sh = torch.empty(N, Lq, M, L, P, 2, **f64), torch.empty(N, Lq, M, L, P, 2, **f64)
        ga, ga_sh = torch.empty(N, Lq, M, L, P, **f64), torch.empty(N, Lq, M, L, P, **f64)
    for n in range(N):
        for m in range(M):
            V = value[n, :, m].double()
            pix = geo["pix"][n, :, m].reshape(Lq, K4)
            w = (bil[n, :, m] * a[n, :, m, :, :, None]).reshape(Lq, K4)
            Vg = V[pix]                                                               # [Lq, 4LP, D]
            out[n, :, m] = torch.einsum("qk,qkd->qd", w, Vg)
            out_sh[n, :, m] = torch.einsum("qk,qkd->qd", w.abs(), Vg.abs())
            if gout is None:
                continue
            go = go_all[n, :, m].double()                                             # [Lq, D]
            T = torch.einsum("qd,qkd->qk", go, Vg).view(Lq, L, P, 4)
            Ta = torch.einsum("qd,qkd->qk", go.abs(), Vg.abs()).view(Lq, L, P, 4)
            b, bx, by, an = bil[n, :, m], dbx[n, :, m], dby[n, :, m], a[n, :, m]
            ga[n, :, m] = (b * T).sum(-1)
            ga_sh[n, :, m] = (b * Ta).sum(-1)
            gl[n, :, m, ..., 0] = an * geo["W"] * (bx * T).sum(-1)
            gl[n, :, m, ..., 1] = an * geo["H"] * (by * T).sum(-1)
            gl_sh[n, :, m, ..., 0] = an.abs() * geo["W"] * (bx.abs() * Ta).sum(-1)
            gl_sh[n, :, m, ..., 1] = an.abs() * geo["H"] * (by.abs() * Ta).sum(-1)
            mk = geo["mask"][n, :, m].reshape(-1)
            idx = pix.reshape(-1)[mk]
            contrib = (w[..., None] * go[:, None, :]).reshape(-1, D)[mk]
            gv[n, :, m].index_add_(0, idx, contrib)
            gv_sh[n, :, m].index_add_(0, idx, contrib.abs())
            cnt = torch.bincount(idx, minlength=S).double()
            gv_c[n, :, m, 0] = (cnt + 4) * U / (1.0 - (cnt + 4) * U)                   # gamma(k + 4)
    u = R.u_out(value.dtype)
    refs["out"] = (out, [(gamma(4 * L * P + 4) * (1 + u), out_sh)])
    if gout is not None:
        c_la = gamma(22 + int(math.log2(locaw_gp(D))))
        refs["grad_value"] = (gv, [(gv_c * (1 + u), gv_sh)])
        refs["grad_loc"] = (gl, [(c_la, gl_sh)])
        refs["grad_attn"] = (ga, [(c_la, ga_sh)])
    return refs


def _ref_rows(ref, N, Lq, L):
    """reference points [*, *, rl, rd] (rows Lq or N Lq, levels 1 or L) -> [N, Lq, 1, L, 1, rd] fp64, as the kernel
    indexes them."""
    rows, rl, rd = ref.shape[0] * ref.shape[1], ref.shape[2], ref.shape[3]
    r = ref.double().reshape(rows, rl, rd)
    r = r.view(1, Lq, rl, rd).expand(N, Lq, rl, rd) if rows == Lq else r.view(N, Lq, rl, rd)
    return r.expand(N, Lq, L, rd)[:, :, None, :, None, :]


def prep_forward_refs(offsets, logits, ref, shapes, N, Lq, M, L, P):
    """softmax over L*P and sampling locations: {"loc": [N, Lq, M, L, P, 2], "attn": [N, Lq, M, L, P]}."""
    dev = offsets.device
    lg = logits.double().view(N, Lq, M, L * P)
    d = lg - lg.amax(-1, keepdim=True)
    attn = torch.softmax(lg, -1)
    delta = U * d.abs() + 4 * U
    c_attn = (delta + delta.amax(-1, keepdim=True) + gamma(L * P + 1)) * (1 + 2.0 ** -20)
    off = offsets.double().view(N, Lq, M, L, P, 2)
    rp = _ref_rows(ref.to(dev), N, Lq, L)
    if rp.shape[-1] == 2:
        wh = torch.tensor([[float(w), float(h)] for h, w in shapes], dtype=torch.float64, device=dev)[:, None, :]
        step = off / wh
        c_loc = 2 * U
    else:
        step = off / P * rp[..., 2:] * 0.5
        c_loc = gamma(2) * (1 + U)
    loc = rp[..., :2] + step
    return {"loc": (loc, [(c_loc, step.abs())]),
            "attn": (attn.view(N, Lq, M, L, P),
                     [(c_attn.view(N, Lq, M, L, P), attn.view(N, Lq, M, L, P)), (1.0, 2.0 ** -147)])}


def prep_backward_refs(gloc, gattn, attn, ref, shapes, out_dtype, N, Lq, M, L, P):
    """{"grad_offsets": [N, Lq, M, L, P, 2], "grad_logits": [N, Lq, M, L, P]} of the prep, in fp64."""
    dev = attn.device
    u = R.u_out(out_dtype)
    a = attn.double().view(N, Lq, M, L * P)
    g = gattn.double().view(N, Lq, M, L * P)
    gl = a * (g - (g * a).sum(-1, keepdim=True))
    gl_sh = a * (g.abs() + (g.abs() * a).sum(-1, keepdim=True))
    glo = gloc.double().view(N, Lq, M, L, P, 2)
    rp = _ref_rows(ref.to(dev), N, Lq, L)
    if rp.shape[-1] == 2:
        wh = torch.tensor([[float(w), float(h)] for h, w in shapes], dtype=torch.float64, device=dev)[:, None, :]
        goff, c_off = glo / wh, gamma(1) * (1 + u)
    else:
        goff, c_off = glo / P * rp[..., 2:] * 0.5, gamma(2) * (1 + u)
    return {"grad_offsets": (goff, [(c_off, goff.abs())]),
            "grad_logits": (gl.view(N, Lq, M, L, P), [(gamma(L * P + 2) * (1 + u), gl_sh.view(N, Lq, M, L, P)),
                                                      (1.0, 2.0 ** -150 + (2.0 ** -134 if u == R.U_BF16 else 2.0 ** -150))])}


# -------------------------------------------------------------------------------------------- the checks
def query_slabs(r):
    """[N, Lq, M, ...] ratios -> worst per (image, head) [N, M]."""
    return r.transpose(1, 2).reshape(r.shape[0], r.shape[2], -1).amax(-1)


def value_slabs(shapes):
    """[N, S, M, D] ratios -> worst per (image, level, head) [N, L, M]."""
    st = level_starts(shapes) + [sum(h * w for h, w in shapes)]
    return lambda r: torch.stack([r[:, st[l]:st[l + 1]].amax((1, 3)) for l in range(len(shapes))], 1)


def check_all(outs, refs, value_dtype, shapes):
    """Reports of every output in `outs` (kernel tensors, any shape that views as the reference's) against `refs`."""
    reps = []
    for name, (ref, terms) in refs.items():
        if name not in outs:
            continue
        u = R.u_out(value_dtype) if name in ("out", "grad_value", "grad_offsets", "grad_logits") else R.U_F32
        block = value_slabs(shapes) if name == "grad_value" else query_slabs
        reps.append(R.check(name, outs[name].reshape(ref.shape), ref, u, terms, block=block))
    return reps


# ------------------------------------------------------------------------------------------------ inputs
def _snap(target, n, reach=48):
    """fp32 normalised coordinates t with pixel coordinate _pix(t, n) == target exactly where one exists within `reach`
    ulps of (target + 0.5) / n, else the nearest of them.  (Not every integer is reachable: x = -1 exactly needs n to be
    a power of two, since (2 t - 1 + 1) lies on a 2^-23 grid.)"""
    t0 = ((target.double() + 0.5) / n).float()
    best, best_err = t0, (_pix(t0, n).double() - target.double()).abs()
    for direction in (math.inf, -math.inf):
        cand = t0
        for _ in range(reach):
            cand = torch.nextafter(cand, torch.full_like(cand, direction))
            err = (_pix(cand, n).double() - target.double()).abs()
            better = err < best_err
            best = torch.where(better, cand, best)
            best_err = torch.where(better, err, best_err)
    return best


PLACEMENTS = ("random", "centre", "integer", "minus_one", "size", "left_strip", "right_strip", "far")


def _coordinate(kind, n, gen):
    """Normalised coordinates along an axis of n pixels for a tensor of placement kinds (indices into PLACEMENTS)."""
    shape = kind.shape
    u = torch.rand(shape, generator=gen, dtype=torch.float64)
    k = torch.randint(0, n, shape, generator=gen).double()
    x = (-1.5 + u * (n + 2.0))                                                   # random: (-1.5, n + 0.5)
    x = torch.where(kind == 1, k + 0.5, x)                                       # pixel centre
    x = torch.where(kind == 2, k, x)                                             # integer: a cell border
    x = torch.where(kind == 3, torch.full_like(x, -1.0), x)                      # outside by exactly nothing
    x = torch.where(kind == 4, torch.full_like(x, float(n)), x)
    x = torch.where(kind == 5, -u * 0.999 - 0.0005, x)                           # (-1, 0): one column in the map
    x = torch.where(kind == 6, n - 1 + 0.0005 + u * 0.999, x)                   # (n - 1, n): likewise
    x = torch.where(kind == 7, torch.where(u < 0.5, -3.0 - u * n, n + 2.0 + u * n), x)
    t = ((x + 0.5) / n).float()
    exact = (kind == 2) | (kind == 3) | (kind == 4)
    return torch.where(exact, _snap(x, n), t)


def sample_locations(gen, N, Lq, M, shapes, P, p_random=0.4):
    """loc [N, Lq, M, L, P, 2]: a fraction p_random of uniform samples over (-1.5, size + 0.5) pixels, the rest spread
    over the special placements (independently for x and y)."""
    L = len(shapes)
    loc = torch.empty(N, Lq, M, L, P, 2)
    for l, (H, W) in enumerate(shapes):
        for ax, n in ((0, W), (1, H)):
            kind = torch.randint(1, len(PLACEMENTS), (N, Lq, M, P), generator=gen)
            kind = torch.where(torch.rand(N, Lq, M, P, generator=gen) < p_random, torch.zeros_like(kind), kind)
            loc[:, :, :, l, :, ax] = _coordinate(kind, n, gen)
    return loc


def attention_weights(gen, N, Lq, M, L, P):
    """softmax rows, with one-hot rows (q % 7 == 0) and rows with zero weights (q % 5 == 0: the even points)."""
    aw = torch.softmax(torch.randn(N, Lq, M, L * P, generator=gen), -1)
    q = torch.arange(Lq)
    hot = torch.randint(0, L * P, (N, Lq, M), generator=gen)
    oh = torch.nn.functional.one_hot(hot, L * P).float()
    aw = torch.where((q % 7 == 0)[None, :, None, None], oh, aw)
    z = (q % 5 == 0)[None, :, None, None] & (torch.arange(L * P) % 2 == 0)
    aw = torch.where(z & (q % 7 != 0)[None, :, None, None], torch.zeros_like(aw), aw)
    return aw.view(N, Lq, M, L, P)


def operands(gen, N, Lq, M, D, shapes, dtype):
    """value [N, S, M, D] and grad_out [N, Lq, M*D] in `dtype`, with an offset and a scale per (image, head, level) of
    the value and per (image, head) of grad_out, so reading another unit's data is an O(1) error in its own slab."""
    S = sum(h * w for h, w in shapes)
    value = torch.randn(N, S, M, D, generator=gen)
    for l, (s0, (h, w)) in enumerate(zip(level_starts(shapes), shapes)):
        n_ = torch.arange(N).view(N, 1, 1, 1)
        m_ = torch.arange(M).view(1, 1, M, 1)
        off = ((3 * n_ + 5 * m_ + 7 * l) % 13 - 6) * 0.5
        sc = 1.0 + ((n_ + 2 * m_ + 3 * l) % 4) * 0.5
        value[:, s0:s0 + h * w] = value[:, s0:s0 + h * w] * sc + off
    gsc = (1.0 + (torch.arange(N).view(N, 1, 1, 1) + torch.arange(M).view(1, 1, M, 1)) % 3)
    gout = (torch.randn(N, Lq, M, D, generator=gen) * gsc + 0.25).reshape(N, Lq, M * D)
    return value.to(dtype), gout.to(dtype)
