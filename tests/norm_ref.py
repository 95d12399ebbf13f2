"""fp64 references with elementwise error bounds for the memory-bound kernels of csrc/norm.cu (LayerNorm forward and
backward, column sums, the LayerScale backward, scale_cols / add / cast) and the depth-wise 3x3 convolution of
csrc/misc.cu, together with the launchers' grid arithmetic that fixes every chain length below.

The rule is tc_ref's (its `check` is used as is): a kernel result passes when, element by element,

    |kernel - ref|  <=  u_out |ref|  +  sum_k c_k shadow_k

with u_out the unit roundoff of the stored type (2^-8 bf16, 2^-24 f32) and each shadow the same expression on absolute
values.  Every reference is evaluated in fp64 on the operands exactly as the kernel reads them (bf16 inputs are exact in
fp32).  The build compiles with nvcc's default FMA contraction, so a multiply-add may or may not be fused: every count
below charges the product its own rounding, which bounds both.

Constants.  u = 2^-24 and gamma(n) = n u / (1 - n u) bounds the relative error of n successive fp32 roundings (Higham,
Accuracy and Stability of Numerical Algorithms, Lemma 3.1); a sum whose every term passes through at most n roundings
errs by at most gamma(n) times the sum of the terms' absolute values.  A chain of k terms is charged k roundings on
every path (its first addition, onto 0, is exact: the count is one high, never low).  A second rounding of a value
that is already off by e adds (1 + u_out) e; the factor (1 + 2^-6) on the constants covers that and the second-order
products of the terms below (all < 2^-12 of the term they multiply).

LayerNorm forward, ln_fwd_kernel<XT, YT, NV> (one warp per row; lane l owns the 4-vectors l + 32 j, j < NV):
  * mean: each lane's `s += ((v0 + v1) + v2) + v3` is a chain of <= 4 NV roundings on any term, the xor butterfly 5
    more (every lane ends with the same value: fp32 addition commutes), the IEEE division by C one ->
    |mu_k - mu| <= dmu = gamma(4 NV + 6) mean|x| (a shadow of the row, not of |mu|: the row's sum may cancel).
  * variance, two-pass: d = x - mu_k (1 rounding), d d (1), the lane chain (4 NV), the butterfly (5), / C (1), + eps
    (1): gamma(4 NV + 9) relative, every term non-negative.  With mu_k = mu + delta, sum (x - mu_k)^2 =
    sum (x - mu)^2 + C delta^2 exactly: the mean's error enters only at second order, delta^2 / (var + eps).
  * rstd: rsqrtf errs by 2 ulp (2^-22 relative) and halves the relative error of its argument ->
    e_rs = gamma(4 NV + 9) / 2 + 2^-22 + dmu^2 / (2 (var + eps)),  rstd: c = e_rs (1 + 2^-6), shadow rstd.
  * y = fma((x - mu_k) rs, g, b): (x - mu_k) = (x - mu) - delta carries the FIRST-order term rs |g| dmu, which dominates
    when |mean| >> std (its shadow scales with mean|x| rs, not with |y|); the rest is three roundings, e_rs and the add:
    y: (gamma(4) + e_rs)(1 + 2^-6) of |xhat g| + 2u |b| + (1 + 2^-6) rs |g| dmu.
LayerNorm backward, ln_bwd2_kernel<DT, XT> with mean and rstd as given inputs (the forward's errors do not enter):
  * xhat = (x - mu) rs: 2 roundings; t = dy g: 1.
  * m1 = sum t / C and m2 = sum t xhat / C: 4 in-thread terms, the 5-level warp butterfly, the 8-term tree (3 levels),
    the product by 1/C (1/C is itself rounded unless C is a power of two: 1 more) -> m1: gamma(15) of A1 = mean|t|,
    m2: gamma(18) of A2 = mean|t xhat| (again the shadows of the sums: m1 and m2 may cancel).
  * dx = rs (t - m1 - xhat m2) + dres: <= 6 more roundings -> c = gamma(24), shadow rs (|t| + A1 + |xhat| A2) + |dres|.
  * dgamma = sum dy xhat, dbeta = sum dy: per-thread chains over the block's rows (block b owns rows 2b, 2b + 1,
    then every 2 grid rows: <= 2 ceil(R / (2 grid)) terms), then reduce_partials<PL> over the grid's partials, then the
    `accumulate` add: gamma(3 + rows + depth + 1) and gamma(rows + depth + 1).
reduce_partials<PL> (PL = 32 iff nparts >= 96): part-lane y sums parts y, y + PL, ... into four accumulators, the
  remainder (<= 3 parts) into the first, so a chain of <= ceil(nparts / 4 PL) + 3 terms; (t0 + t1) + (t2 + t3): 2; the
  PL-term chain over the part-lanes: PL -> depth(nparts) = ceil(nparts / 4 PL) + 5 + PL.
colsum_kernel<XT, YT, kMul>: thread (lane, ty) of row block y sums rows y 8 + ty, + 8 rb, ... in row order (the
  four-rows-in-flight loop adds them in the same order): ceil(M / (8 rb)) terms, one product rounding (bf16 x bf16 is
  exact in fp32, f32 x f32 is not unless contracted: always charged), the 8-term chain over ty, depth(rb), accumulate:
  c = gamma(ceil(M / 8 rb) + 1 + 8 + depth(rb) + 1), shadow sum |X Y| (+ |prior|).
layerscale_bwd_kernel<UT>: du = (d g).to(UT) is one fp32 product and one store rounding, exactly as torch computes it:
  compared bit for bit.  dgamma = sum d u (u as read), dbias = sum du as stored: the colsum chains with rb =
  colsum_rb(M) row blocks.
scale_cols / add / cast: one fp32 operation and the store: bit for bit against torch's fp32 operation and .to(out).
Depth-wise 3x3 convolution (one thread per (image, token, 4 channels)):
  * forward: acc = bias + a chain of <= 9 products (the taps inside the map, in tap order): c_pre = gamma(10) of
    S = |bias| + sum |w| |x|; `pre` is stored in T.  The fused GELU is evaluated on the fp32 acc: 0.5 x (1 + erff(x /
    sqrt 2)) with erff within 2 ulp (<= 2^-23 absolute below 1), the argument's rounding (<= 0.48 u of erf's change),
    the add and the product (u |y| <= u |x|) -> <= 3.8 u |x|: C_GELU = 4 u with shadow |x| -- not |gelu(x)|: for
    x << 0, 1 + erff(x / sqrt 2) cancels.  y = gelu: (GELU_LIP + 2^-6) c_pre S + C_GELU |pre|.
  * backward: g = dy GELU'(pre) from the STORED pre.  dgelu_erf = cdf + x 0.3989 __expf(-x x / 2): cdf as above
    (<= 2.74 u), __expf within 2 + floor(1.173 |a|) ulp at a = x^2 / 2 (<= (4 + 2.35 a) u relative), the rounded
    argument (a u), the constant and two products (3 u), the add (<= 1.13 u); with max x phi(x) = 0.242 and
    max x^3 phi(x) = 0.463: <= 6.4 u absolute -> C_DGELU = 8 u.  g = dy GELU' (1 product) is stored in T before the
    convolution reads it: E_g = (u + u_T)(1 + 2^-6) |g| + C_DGELU (1 + 2^-6) |dy| (0 when not fused: g = dy as read).
  * dx = a chain of <= 9 products of g at the neighbours, stored in T: gamma(10) (1 + 2^-6) of sum |w| |g| +
    (1 + 2^-6) sum |w| E_g.
  * dweight, dbias: per-thread chains over ceil(rows / (8 rb)) tokens (+ 1 product), the 8-term chain, then
    dwconv_reduce_kernel's sequential chain over the rb partials, accumulate: gamma(rows + 1 + 8 + rb + 1) of
    sum |g| |x| (sum |g|), plus sum E_g |x| (sum E_g).

Slabs: the LayerNorm outputs report their worst ratio per row block, column sums and parameter gradients per
128-column block, the convolution per (image, map) and per 128-channel block -- so a unit that went wrong is named.
"""
import torch

import tc_ref as R

U = R.U_F32
SLACK = 1.0 + 2.0 ** -6
C_GELU = 4 * U
C_DGELU = 8 * U


def gamma(n):
    return n * U / (1.0 - n * U)


# ---------------------------------------------------------------------------------- the launchers' arithmetic
LN_FWD_ROWS = 8               # rows (warps) per ln_fwd block
LN_BWD_ROWS = 2               # rows per ln_bwd2 block iteration
LN_BWD_BLOCKS = 4 * 148       # persistent blocks of the LayerNorm backward


def ln_nv(C):
    nv = -(-C // 128)
    for k in (1, 2, 3, 4, 6, 8):
        if nv <= k:
            return k
    raise ValueError(C)


def ln_fwd_grid(R_):
    return -(-R_ // LN_FWD_ROWS)


def ln_bwd_grid(R_):
    return min(-(-R_ // LN_BWD_ROWS), LN_BWD_BLOCKS)


def reduce_pl(nparts):
    return 32 if nparts >= 96 else 8


def reduce_depth(nparts):
    pl = reduce_pl(nparts)
    return -(-nparts // (4 * pl)) + 5 + pl


def colsum_rb(M, N=1 << 30):
    cb = -(-N // 128)
    want = 1024 // cb if cb < 8 else 128
    return max(1, min(-(-M // 64), want))


def dwconv_fwd_grid(B, ntok, C):
    return -(-(B * ntok * (C // 4)) // 1024)


def dwconv_row_blocks(rows, C):
    return max(1, min(-(-rows // 64), max(1, 296 // -(-C // 128))))


# ------------------------------------------------------------------------------------------------ slabs
def row_slabs(rows):
    """Worst ratio per block of `rows` rows (of a [R, C] or [R] output)."""
    return lambda r: R.slab_max(r, (rows,) + tuple(r.shape[1:])).reshape(-1)


def col_slabs(r):
    """Worst ratio per 128-column block of a [N] or [N, k] output."""
    return R.slab_max(r, (128,) + tuple(r.shape[1:]))


def dw_slabs(maps):
    """[B, ntok, C] -> [B, n_maps, ceil(C / 128)]: the worst ratio per (image, map, 128-channel block)."""
    def f(r):
        out, s = [], 0
        for h, w in maps:
            out.append(R.slab_max(r[:, s:s + h * w], (1, h * w, 128))[:, 0])
            s += h * w
        return torch.stack(out, 1)
    return f


# ------------------------------------------------------------------------------------------- LayerNorm
def ln_fwd_ref(x, g, b, eps, nv):
    """{"y", "mean", "rstd"}: (ref, [(c, shadow), ...]) of LayerNorm over the last dim of x [R, C] (x as read)."""
    x64, g64, b64 = x.double(), g.double(), b.double()
    mu = x64.mean(1)
    xc = x64 - mu[:, None]
    var = (xc * xc).mean(1)
    rs = 1.0 / torch.sqrt(var + eps)
    dmu = gamma(4 * nv + 6) * x64.abs().mean(1)
    e_rs = gamma(4 * nv + 9) / 2 + 4 * U + dmu * dmu / (2 * (var + eps))
    xg = xc * rs[:, None] * g64
    y = xg + b64
    return {"y": (y, [((gamma(4) + e_rs[:, None]) * SLACK, xg.abs()), (2 * U, b64.abs().expand_as(y)),
                      (SLACK, (rs * dmu)[:, None] * g64.abs())]),
            "mean": (mu, [(1.0, dmu)]),
            "rstd": (rs, [(e_rs * SLACK, rs)])}


def ln_bwd_ref(dy, x, g, mu, rs, dres=None, grid=None, prior_g=None, prior_b=None):
    """{"dx", "dgamma", "dbeta"} of the LayerNorm backward with mean / rstd given (f32, as the kernel reads them).
    `grid`: the kernel's block count (chain lengths of the column partials); prior_*: the values `accumulate` adds to."""
    R_, C = x.shape
    grid = grid or ln_bwd_grid(R_)
    dy64, x64, g64 = dy.double(), x.double(), g.double()
    rs64 = rs.double()[:, None]
    xh = (x64 - mu.double()[:, None]) * rs64
    t = dy64 * g64
    m1, m2 = t.mean(1, keepdim=True), (t * xh).mean(1, keepdim=True)
    a1, a2 = t.abs().mean(1, keepdim=True), (t * xh).abs().mean(1, keepdim=True)
    dx = rs64 * (t - m1 - xh * m2)
    sh = rs64 * (t.abs() + a1 + xh.abs() * a2)
    if dres is not None:
        dx, sh = dx + dres.double(), sh + dres.double().abs()
    rows = LN_BWD_ROWS * -(-R_ // (LN_BWD_ROWS * grid))
    depth = reduce_depth(grid)
    dg, dgs = (dy64 * xh).sum(0), (dy64 * xh).abs().sum(0)
    db, dbs = dy64.sum(0), dy64.abs().sum(0)
    if prior_g is not None:
        dg, dgs = dg + prior_g.double(), dgs + prior_g.double().abs()
    if prior_b is not None:
        db, dbs = db + prior_b.double(), dbs + prior_b.double().abs()
    return {"dx": (dx, [(gamma(24), sh)]),
            "dgamma": (dg, [(gamma(3 + rows + depth + 1), dgs)]),
            "dbeta": (db, [(gamma(rows + depth + 1), dbs)])}


# ---------------------------------------------------------------------------------------- column sums
def colsum_ref(X, Y=None, rb=None, prior=None):
    """sum over rows of X (X * Y) [M, N] (the logical views, as read), with `rb` row blocks."""
    M, N = X.shape
    rb = rb or colsum_rb(M, N)
    p = X.double() if Y is None else X.double() * Y.double()
    ref, sh = p.sum(0), p.abs().sum(0)
    if prior is not None:
        ref, sh = ref + prior.double(), sh + prior.double().abs()
    c = gamma(-(-M // (8 * rb)) + 1 + 8 + reduce_depth(rb) + 1)
    return ref, [(c, sh)]


def layerscale_ref(d, u, g, du_kernel_dtype):
    """{"du": exact tensor (torch's rounding), "dgamma", "dbias"}; u is None when dgamma is not asked for."""
    M, N = d.shape
    du = (d.float() * g.float()).to(du_kernel_dtype)
    rb = colsum_rb(M)
    r = {"du": du, "dbias": colsum_ref(du, None, rb)}
    if u is not None:
        r["dgamma"] = colsum_ref(d, u, rb)
    return r


# ------------------------------------------------------------------------------------ depth-wise convolution
def _maps(t, maps):
    """[B, ntok, C] -> [(start, h, w, view [B, h, w, C])]."""
    out, s = [], 0
    for h, w in maps:
        out.append((s, h, w, t[:, s:s + h * w].reshape(t.shape[0], h, w, t.shape[2])))
        s += h * w
    return out


def _shift(t, oy, ox):
    """t [B, h, w, C] -> s with s[p] = t[p + (oy, ox)], zero outside the map."""
    _, h, w, _ = t.shape
    p = torch.nn.functional.pad(t, (0, 0, 1, 1, 1, 1))
    return p[:, 1 + oy:1 + oy + h, 1 + ox:1 + ox + w]


TAPS = [(j // 3 - 1, j % 3 - 1) for j in range(9)]


def dwconv_fwd_ref(x, weight, bias, maps, fuse, dtype):
    """{"pre": ..., "y": ...} of the depth-wise 3x3 convolution (+ GELU) on token-major x [B, ntok, C] (as read)."""
    B, ntok, C = x.shape
    w9 = weight.double().reshape(C, 9)
    b64 = bias.double()
    acc = torch.empty(B, ntok, C, dtype=torch.float64, device=x.device)
    S = torch.empty_like(acc)
    for s, h, w, xm in _maps(x.double(), maps):
        a = b64.expand(B, h, w, C).clone()
        sa = b64.abs().expand(B, h, w, C).clone()
        for j, (oy, ox) in enumerate(TAPS):
            v = _shift(xm, oy, ox)
            a += w9[:, j] * v
            sa += w9[:, j].abs() * v.abs()
        acc[:, s:s + h * w] = a.reshape(B, h * w, C)
        S[:, s:s + h * w] = sa.reshape(B, h * w, C)
    c = gamma(10)
    r = {"pre": (acc, [(c * SLACK, S)])}
    if fuse:
        r["y"] = (R._gelu(acc), [((R.GELU_LIP + 2.0 ** -6) * c, S), (C_GELU * SLACK, acc.abs())])
    else:
        r["y"] = r["pre"]
    return r


def dwconv_bwd_ref(dy, pre, x, weight, maps, fuse, dtype, rb, prior_w=None, prior_b=None):
    """{"dx", "dweight" [C, 9], "dbias"} of the depth-wise 3x3 convolution with g = dy (unfused) or dy GELU'(pre)
    (pre as stored); `rb`: the backward's row blocks."""
    B, ntok, C = x.shape
    dy64 = dy.double()
    if fuse:
        g = dy64 * R._dgelu(pre.double())
        eg = (U + R.u_out(dtype)) * SLACK * g.abs() + C_DGELU * SLACK * dy64.abs()
    else:
        g, eg = dy64, torch.zeros_like(dy64)
    w9 = weight.double().reshape(C, 9)
    dx = torch.empty_like(g)
    sdx, edx = torch.empty_like(g), torch.empty_like(g)
    dw = torch.zeros(C, 9, dtype=torch.float64, device=x.device)
    sdw, edw = torch.zeros_like(dw), torch.zeros_like(dw)
    x64 = x.double()
    for (s, h, w, gm), (_, _, _, em), (_, _, _, xm) in zip(_maps(g, maps), _maps(eg, maps), _maps(x64, maps)):
        a, sa, ea = torch.zeros_like(gm), torch.zeros_like(gm), torch.zeros_like(gm)
        for j, (oy, ox) in enumerate(TAPS):
            gs, es = _shift(gm, -oy, -ox), _shift(em, -oy, -ox)
            a += w9[:, j] * gs
            sa += w9[:, j].abs() * gs.abs()
            ea += w9[:, j].abs() * es
            xs = _shift(xm, oy, ox)
            dw[:, j] += (gm * xs).sum((0, 1, 2))
            sdw[:, j] += (gm.abs() * xs.abs()).sum((0, 1, 2))
            edw[:, j] += (em * xs.abs()).sum((0, 1, 2))
        dx[:, s:s + h * w] = a.reshape(B, h * w, C)
        sdx[:, s:s + h * w] = sa.reshape(B, h * w, C)
        edx[:, s:s + h * w] = ea.reshape(B, h * w, C)
    db, sdb, edb = g.sum((0, 1)), g.abs().sum((0, 1)), eg.sum((0, 1))
    if prior_w is not None:
        dw, sdw = dw + prior_w.double().reshape(C, 9), sdw + prior_w.double().reshape(C, 9).abs()
    if prior_b is not None:
        db, sdb = db + prior_b.double(), sdb + prior_b.double().abs()
    cp = gamma(-(-(B * ntok) // (8 * rb)) + 1 + 8 + rb + 1)
    return {"dx": (dx, [(gamma(10) * SLACK, sdx), (SLACK, edx)]),
            "dweight": (dw, [(cp, sdw), (1 + cp, edw)]),
            "dbias": (db, [(cp, sdb), (1 + cp, edb)])}
