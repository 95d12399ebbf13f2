"""fp64 references with elementwise error bounds for the bf16 tensor-core kernels (GEMM epilogues, attention
forward / backward, implicit 3x3 convolution), and the host simulation of the attention forward's lazy rescaling.

Every reference is evaluated in fp64 on the same bf16-rounded operands the kernel reads, together with one or
more ABSOLUTE-VALUE SHADOWS: the same expression on |operands| (|A||B|^T, P|V|, |P|^T|dO|, ...).  A kernel result
passes when, element by element,

    |kernel - ref|  <=  u_out |ref|  +  sum_k c_k shadow_k

  u_out   the unit roundoff of the stored output: 2^-8 for bf16 (8 significant bits: a correctly rounded value
          can be off by half a spacing = 2^-8 of itself just above a power of two) and 2^-24 for f32.
          (A rounding of a value that is itself off by e adds (1 + u_out) e: the constants below absorb the factor.)
  c_k     derived from where the kernel rounds -- never fitted to measurements:
  * tensor-core accumulation: the products of bf16 operands are exact in fp32; each tcgen05.mma step of K = 16 adds
    16 products and the running fp32 accumulator with the addends aligned to the largest one and one truncation to
    fp32 (<= 2^-23 relative, doubled for the alignment) -> C_MMA(K) = (ceil(K / 16) + 4) 2^-22 of |A||B|^T (the +4:
    the in-step adder tree of 16 terms);
  * split-K: one more fp32 rounding (red.global.add) per split;
  * epilogue: bias add, LayerScale FMA, residual add, and GELU / GELU' from the Abramowitz-Stegun erfc
    (|error| <= 1.5e-7 < 2^-22) with rcp.approx / ex2.approx (<= 2^-22 relative each): 8 more units of 2^-22;
  * attention: P and dS are rounded to bf16 before their MMAs (2^-8 relative each); ex2.approx (2^-22 relative);
    the log2-domain argument s log2(e) / 8 - m is formed by one fmaf (2^-24 of |s log2(e) / 8| + |m|) -- an error
    of d in the exponent is a relative error of ln(2) d of the exponential, shared by numerator and denominator;
    l (the fp32 row sum of the UNROUNDED exponentials) passes through <= 18 + 2 nkv additions / rescales;
    the backward recomputes P from the kernel's lse (its error is the forward's lse bound) and reads
    D = rowsum(dO o O) from the kernel's bf16 O (its error is |dO| times the forward's bound on O).
The exact quantities (which terms, which shadows) are written next to each reference below.

`check` returns the largest err / bound ratio, where it is and the largest ratio of every slab (an output tile of
the GEMM, an (image, head) of the attention), so a failure names the unit that went wrong.
"""
import json
import math
import os
import tempfile

import torch

U_BF16 = 2.0 ** -8
U_F32 = 2.0 ** -24
LOG2E = 1.0 / math.log(2.0)
SCALE = 64 ** -0.5          # head_dim 64 (exact power of two)
TILE = 128                  # attention forward: query / key tile


def u_out(dtype):
    return U_BF16 if dtype == torch.bfloat16 else U_F32


def c_mma(k, splits=1):
    """fp32 tensor-core accumulation of a k-long bf16 dot product (split-K: `splits` partial sums added in fp32)."""
    return (math.ceil(k / 16) + 4 + splits) * 2.0 ** -22


C_EPI = 8 * 2.0 ** -22      # roundings and function approximations of the fused GEMM epilogue


# -------------------------------------------------------------------------------------------- the check
class Report:
    def __init__(self, name, ratio, where, err, bound, ref, out, slabs):
        self.name, self.ratio, self.where, self.err, self.bound, self.ref, self.out, self.slabs = \
            name, ratio, where, err, bound, ref, out, slabs

    @property
    def ok(self):
        return self.ratio <= 1.0

    def __str__(self):
        s = (f"{self.name}: max err/bound {self.ratio:.3g} at {self.where} (kernel {self.out:.6g}, ref {self.ref:.6g}, "
             f"err {self.err:.3g}, bound {self.bound:.3g})")
        if self.slabs is not None and not self.ok:
            bad = (self.slabs > 1).nonzero().tolist()
            s += f"; {len(bad)} of {self.slabs.numel()} slabs over their bound, first {bad[:8]}"
        return s


def slab_max(r, block):
    """amax of `r` over blocks of shape `block` (one entry per dimension; the last block of a dimension may be short)."""
    pad = []
    for n, b in zip(reversed(r.shape), reversed(block)):
        pad += [0, (-n) % b]
    r = torch.nn.functional.pad(r, pad, value=0.0)
    shape = []
    for n, b in zip(r.shape, block):
        shape += [n // b, b]
    r = r.reshape(shape)
    return r.amax(dim=tuple(range(1, 2 * len(block), 2)))


def check(name, out, ref, u, terms, block=None):
    """Elementwise |out - ref| <= u |ref| + sum c * shadow over `terms` = [(c, shadow), ...] (c and shadow broadcast
    against ref).  Non-finite kernel values count as an infinite ratio.  `block`: the slab shape for slab_max, or a
    function from the ratio tensor to the per-slab maxima."""
    out64 = out.detach().to(device=ref.device, dtype=torch.float64)
    err = (out64 - ref).abs()
    bound = u * ref.abs()
    for c, s in terms:
        bound = bound + c * s
    ratio = err / bound.clamp_min(1e-300)
    ratio = torch.where(err == 0, torch.zeros_like(ratio), ratio)
    ratio = torch.where(torch.isfinite(out64), ratio, torch.full_like(ratio, math.inf))
    i = int(ratio.flatten().argmax())
    where = tuple(int(x) for x in torch.unravel_index(torch.tensor(i), ratio.shape))
    slabs = None if block is None else (block(ratio) if callable(block) else slab_max(ratio, block)).cpu()
    return Report(name, float(ratio.flatten()[i]), where, float(err.flatten()[i]), float(bound.flatten()[i]),
                  float(ref.flatten()[i]), float(out64.flatten()[i]), slabs)


# ---------------------------------------------------------------------------------------------- the trace
def traced(fn):
    """Run fn under torch.profiler; return (its result, [(kernel name, grid)] of the project's kernels)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        r = fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            ev = json.load(f)["traceEvents"]
    ks = [(e["name"].replace(" ", "").replace("(int)", ""), tuple(e.get("args", {}).get("grid", ()))) for e in ev
          if e.get("cat") == "kernel" and "asis::" in e.get("name", "")]
    return r, ks


def expect_kernel(ks, pattern, grid):
    """The one launch whose name contains `pattern` (spaces ignored) and its grid == `grid` (a tuple)."""
    pat = pattern.replace(" ", "")
    hits = [k for k in ks if pat in k[0]]
    assert len(hits) == 1, f"expected one launch of {pattern}, trace has {[k[0] for k in ks]}"
    name, g = hits[0]
    assert g, f"the trace records no grid for {name}"
    assert tuple(g) + (1,) * (3 - len(g)) == tuple(grid) + (1,) * (3 - len(grid)), (name, g, grid)
    return name


# -------------------------------------------------------------------------------------- the output guards
NAN_BITS = {2: 0x7fcb, 4: 0x7fc00bad}
GUARD = 64


def bits(t):
    return t.view(torch.int16 if t.element_size() == 2 else torch.int32)


def guarded(shape, dtype, device="cuda"):
    """(buffer, view): `view` of `shape` inside a NaN-filled buffer with GUARD elements on each side."""
    n = math.prod(shape)
    buf = torch.empty(n + 2 * GUARD, dtype=dtype, device=device)
    bits(buf).fill_(NAN_BITS[buf.element_size()])
    return buf, buf[GUARD:GUARD + n].view(shape)


def guards_intact(buf):
    b = bits(buf)
    nan = NAN_BITS[buf.element_size()]
    return bool((b[:GUARD] == nan).all()) and bool((b[-GUARD:] == nan).all())


# ------------------------------------------------------------------------------------------------- GEMM
def _gelu(h):
    return 0.5 * h * (1.0 + torch.erf(h * 0.5 ** 0.5))


def _dgelu(h):
    return 0.5 * (1.0 + torch.erf(h * 0.5 ** 0.5)) + h * torch.exp(-0.5 * h * h) / math.sqrt(2 * math.pi)


GELU_LIP = 1.13             # max |GELU'| (at x = 2^0.5); max |GELU''| = 0.80 < 1


def gemm_ref(A, B, epilogue="none", bias=None, gamma=None, residual=None, aux=None, c_old=None, splits=1):
    """C = epi(A B^T) with A [M, K], B [N, K] (the logical, K-contiguous views of the operands), in fp64.
    Returns {output name: (ref, [(c, shadow), ...])}; output names: "c" and, where the epilogue writes one, "aux".
      none            c = acc + bias                      shadow S + |bias|            (S = |A||B|^T)
      gelu            c = gelu(h), h = acc + bias         shadow 1.13 (S + |bias|)     aux = h: S + |bias|
      gelu_grad       c = gelu(h), aux = gelu'(h)         aux: S + |bias| + 1 (the erfc approximation's absolute error)
      scale_residual  c = res + gamma h, aux = h          shadow |res| + |gamma| (S + |bias|)
      dgelu           c = acc gelu'(aux)                  shadow S (|gelu'(aux)| + 1)
      mul_aux         c = acc aux                         shadow S |aux|
      accumulate      c = c_old + acc                     shadow |c_old| + S
    The c of every shadow is c_mma(K, splits) + C_EPI."""
    A64, B64 = A.double(), B.double()
    acc = A64 @ B64.t()
    S = A64.abs() @ B64.abs().t()
    c = c_mma(A.shape[1], splits) + C_EPI
    b = bias.double() if bias is not None else torch.zeros(B.shape[0], dtype=torch.float64, device=A.device)
    h, Sh = acc + b, S + b.abs()
    if epilogue == "none":
        return {"c": (h, [(c, Sh)])}
    if epilogue == "gelu":
        return {"c": (_gelu(h), [(c, GELU_LIP * Sh)]), "aux": (h, [(c, Sh)])}
    if epilogue == "gelu_grad":
        return {"c": (_gelu(h), [(c, GELU_LIP * Sh)]), "aux": (_dgelu(h), [(c, Sh + 1.0)])}
    if epilogue == "scale_residual":
        g, r = gamma.double(), residual.double()
        return {"c": (r + g * h, [(c, r.abs() + g.abs() * Sh)]), "aux": (h, [(c, Sh)])}
    if epilogue == "dgelu":
        d = _dgelu(aux.double())
        return {"c": (acc * d, [(c, S * (d.abs() + 1.0))])}
    if epilogue == "mul_aux":
        x = aux.double()
        return {"c": (acc * x, [(c, S * x.abs())])}
    if epilogue == "accumulate":
        o = c_old.double()
        return {"c": (o + acc, [(c, o.abs() + S)])}
    raise ValueError(epilogue)


# -------------------------------------------------------------------------------------------- attention
def _split_qkv(qkv, H):
    Bn, T, _ = qkv.shape
    x = qkv.double().view(Bn, T, 3, H, 64).permute(2, 0, 3, 1, 4)        # [3, B, H, T, 64]
    return x[0], x[1], x[2]


def attention_forward_ref(qkv, H):
    """out [B, T, H*64] and lse [B, H, T] of softmax(q k^T / 8) v, plus their bounds, and the softmax pieces the
    backward reference reuses.
      out: u_out = 2^-8 (bf16 store); shadow P|V| with c_O = 2^-8 (bf16 P) + 2 delta + c_mma(T) + c_l + 2^-22 (1/l)
      lse: absolute, delta + c_l + 2^-22 (|m| log2 e + |log2 l| + 2) ln 2   (log2f, the sum and the ln 2 product)
    where, per row, delta = ln 2 (c_mma(64) max_j (|q||k|^T)_j log2(e) / 8 + 2^-24 (2 max_j |s_j| log2 e)) + 2 2^-22
    is the relative error of one exponential (score MMA, the fmaf of the exponent, ex2.approx and the rescale factor)
    and c_l = (18 + 2 nkv) 2^-24 the relative error of the fp32 row sum l."""
    q, k, v = _split_qkv(qkv, H)
    Bn, T = qkv.shape[0], qkv.shape[1]
    nkv = (T + TILE - 1) // TILE
    s = (q @ k.transpose(-1, -2)) * SCALE
    sa = (q.abs() @ k.abs().transpose(-1, -2)) * SCALE
    m = s.amax(-1, keepdim=True)
    e = torch.exp(s - m)
    l = e.sum(-1, keepdim=True)
    P = e / l
    O = P @ v
    Oa = P @ v.abs()
    lse = (m + torch.log(l)).squeeze(-1)
    delta = math.log(2) * (c_mma(64) * sa.amax(-1) * LOG2E + 2 * U_F32 * s.abs().amax(-1) * LOG2E) + 2 * 2.0 ** -22
    c_l = (18 + 2 * nkv) * U_F32
    c_o = U_BF16 + 2 * delta + c_mma(T) + c_l + 2.0 ** -22                                    # [B, H, T]
    lse_abs = delta + c_l + 2.0 ** -22 * (m.squeeze(-1).abs() * LOG2E + torch.log2(l.squeeze(-1)) + 2) * math.log(2)

    def bhtd(t):                                                                              # [B,H,T,64] -> [B,T,H*64]
        return t.permute(0, 2, 1, 3).reshape(Bn, T, H * 64)

    out_bound_terms = [(bhtd(c_o.unsqueeze(-1).expand_as(Oa)), bhtd(Oa))]
    return dict(out=(bhtd(O), out_bound_terms), lse=(lse, [(1.0, lse_abs)]),
                _P=P, _delta=delta, _lse_abs=lse_abs, _q=q, _k=k, _v=v, _O=O)


def attention_backward_ref(qkv, H, dout, fwd, out_kernel):
    """dqkv [B, T, 3*H*64] = d/dqkv of <out, dout> with the standard softmax backward in fp64
    (dV = P^T dO, dP = dO V^T, D = rowsum(dO o O), dS = P o (dP - D), dQ = dS K / 8, dK = dS^T Q / 8), and its bound.
    The kernel's P carries a relative error delta_b = delta + |lse error| (it is recomputed from the kernel's lse) and
    is rounded to bf16; its D is formed from the kernel's bf16 O: |D' - D| <= D_err = |dO| . bound(O) + 2^-18 |dO||O|.
    dS (bf16) then errs by (2^-8 + delta_b + 2^-23) |dS| + P o (c_mma(64) |dO||V|^T + D_err), so
      dV: c = 2^-8 + delta_b + c_mma(T)               shadow P^T |dO|
      dQ: c = 2^-8 + delta_b + 2^-23 + c_mma(T)       shadow |dS| |K| / 8;   c = 1, shadow E |K| / 8
      dK: likewise with |dS|^T |Q| / 8 and E^T |Q| / 8,   E = P o (c_mma(64) |dO||V|^T + D_err)
    delta_b is taken per (image, head) (its largest row)."""
    P, q, k, v, O = fwd["_P"], fwd["_q"], fwd["_k"], fwd["_v"], fwd["_O"]
    Bn, T = qkv.shape[0], qkv.shape[1]
    dO = dout.double().view(Bn, T, H, 64).permute(0, 2, 1, 3)
    Ok = out_kernel.double().view(Bn, T, H, 64).permute(0, 2, 1, 3)
    (oref, [(c_o, oa)]) = fwd["out"]
    o_bound = (U_BF16 * oref.abs() + c_o * oa).view(Bn, T, H, 64).permute(0, 2, 1, 3)
    dV = P.transpose(-1, -2) @ dO
    dP = dO @ v.transpose(-1, -2)
    D = (dO * O).sum(-1, keepdim=True)
    dS = P * (dP - D)
    dQ = dS @ k * SCALE
    dK = dS.transpose(-1, -2) @ q * SCALE
    D_err = (dO.abs() * o_bound).sum(-1, keepdim=True) + 2.0 ** -18 * (dO.abs() * Ok.abs()).sum(-1, keepdim=True)
    E = P * (c_mma(64) * (dO.abs() @ v.abs().transpose(-1, -2)) + D_err)
    dSa = dS.abs()
    delta_b = (fwd["_delta"] + fwd["_lse_abs"]).amax(-1)[..., None, None]                  # [B, H, 1, 1]
    c_v = U_BF16 + delta_b + c_mma(T)
    c_s = U_BF16 + delta_b + 2.0 ** -23 + c_mma(T)

    def pack(dq, dk, dv):                                                                     # -> [B, T, 3*H*64]
        return torch.stack([dq, dk, dv], 0).permute(1, 3, 0, 2, 4).reshape(Bn, T, 3 * H * 64)

    z = torch.zeros_like(dQ)
    ref = pack(dQ, dK, dV)
    sh_main = pack(dSa @ k.abs() * SCALE, dSa.transpose(-1, -2) @ q.abs() * SCALE, P.transpose(-1, -2) @ dO.abs())
    c_main = pack(c_s.expand_as(dQ), c_s.expand_as(dK), c_v.expand_as(dV))
    sh_e = pack(E @ k.abs() * SCALE, E.transpose(-1, -2) @ q.abs() * SCALE, z)
    return ref, [(c_main, sh_main), (1.0, sh_e)]


def rescale_sim(qkv, H):
    """The forward kernel's lazy-rescaling decision per row and key tile, simulated on the host (log2 domain: the first
    key tile sets the running maximum m; tile j > 0 rescales O and l when max_j(s) log2(e) - m > 8 and then moves m).
    Returns (fires [B, H, T, nkv] bool, margin [B, H, T]: the smallest |growth - 8| of any decision, for rows whose
    decision could flip under the kernel's fp32 scores)."""
    q, k, _ = _split_qkv(qkv, H)
    T = qkv.shape[1]
    nkv = (T + TILE - 1) // TILE
    s = (q @ k.transpose(-1, -2)) * (SCALE * LOG2E)
    tm = torch.stack([s[..., j * TILE:min(T, (j + 1) * TILE)].amax(-1) for j in range(nkv)], -1)
    m = tm[..., 0].clone()
    fires = torch.zeros(tm.shape, dtype=torch.bool, device=tm.device)
    margin = torch.full_like(m, math.inf)
    for j in range(1, nkv):
        grow = torch.maximum(m, tm[..., j]) - m
        fires[..., j] = grow > 8.0
        margin = torch.minimum(margin, (grow - 8.0).abs())
        m = torch.where(fires[..., j], tm[..., j], m)
    return fires, margin


RAMP_R = 40.0              # ramp of the key levels (natural units of score: a_i R / 8 over the whole row)


def attention_inputs(kind, Bn, T, H, gen):
    """qkv [B, T, 3*H*64] (fp32 values representable in bf16; call .bfloat16()) for the accuracy cases.
    Every (image, head) gets its own V offset, so a unit that reads another unit's data is off by O(1).
      randn  N(0, 1) q, k, v: scores of sigma ~ 1, no rescale fires
      ramp   q_i = a_i u, k_j = level(j) R / nkv u (u = 1/8 in every channel, so s_ij = a_i level(j) R / (8 nkv)):
             the level is the key tile index, and the last valid key sits one level above the last tile -- later tiles
             out-score earlier ones by up to a R / 8 = 200 natural units, several times in one row, in the masked last
             tile, also when T <= 128 or the last tile holds one key; a_i in [-A/4, A] (a < 0: the first tile holds the
             maximum, a ~ 0: near-uniform rows); rows t % 17 == 0 have q = 0 exactly (uniform softmax: mean(V))
      sub    like ramp with a_i in [0, a_sub]: total growth <= 7.5 log2 units, so P reaches ~2^7.5 with no rescale
      qzero  N(0, 1) k, v; q = 0 on rows t % 3 == 0 (exactly uniform rows)"""
    nkv = (T + TILE - 1) // TILE
    q = torch.randn(Bn, T, H, 64, generator=gen)
    k = torch.randn(Bn, T, H, 64, generator=gen)
    v = torch.randn(Bn, T, H, 64, generator=gen)
    t = torch.arange(T)
    if kind in ("ramp", "sub"):
        level = (t // TILE).double()
        level[T - 1] = nkv
        r = level * RAMP_R / nkv
        frac = torch.frac(torch.arange(Bn * H * T, dtype=torch.float64) * 0.6180339887).view(Bn, H, T).permute(0, 2, 1)
        if kind == "ramp":
            a = 1600.0 / RAMP_R * (1.25 * frac - 0.25)
        else:
            a = 7.5 * math.log(2) * 8 / RAMP_R * frac
        a[:, t % 17 == 0] = 0.0
        u = torch.full((64,), 0.125, dtype=torch.float64)
        q = (a[..., None] * u).float()
        k = (r[None, :, None, None] * u).float().expand(Bn, T, H, 64).contiguous()
    elif kind == "qzero":
        q[:, t % 3 == 0] = 0.0
    elif kind != "randn":
        raise ValueError(kind)
    off = (torch.arange(Bn * H).view(Bn, 1, H, 1) % 11 - 5) * 0.5
    v = v + off
    return torch.stack([q, k, v], 2).reshape(Bn, T, 3 * H * 64).bfloat16().float()


def attn_units(Bn, T, H, sms):
    """The forward launcher's arithmetic: items = pairs of 128-query tiles of one (image, head), grid = min(items, SMs);
    CTA c takes items c, c + grid, ..."""
    npair = ((T + TILE - 1) // TILE + 1) // 2
    items = npair * H * Bn
    return items, min(items, sms), npair


# ----------------------------------------------------------------------------------------- convolution
def conv3x3_ref(x, w, bias=None, dy=None):
    """3x3 / stride 1 / pad 1 convolution on the logical (unpadded) NCHW maps in fp64 and its two gradients.
    x [B, Cin, H, W], w [Cout, Cin, 3, 3], dy [B, Cout, H, W]; products of bf16 values, K = 9 Cin / 9 Cout / B H W.
    Returns {"y": (ref, shadow), "dx": ..., "dw": ...} with shadows on |operands| (y: + |bias|); c = c_mma(K)."""
    F = torch.nn.functional
    x64, w64 = x.double(), w.double()
    b64 = bias.double() if bias is not None else None
    r = {"y": (F.conv2d(x64, w64, b64, padding=1),
               F.conv2d(x64.abs(), w64.abs(), b64.abs() if b64 is not None else None, padding=1))}
    if dy is not None:
        dy64 = dy.double()
        r["dx"] = (F.conv_transpose2d(dy64, w64, padding=1), F.conv_transpose2d(dy64.abs(), w64.abs(), padding=1))
        gw = torch.nn.grad.conv2d_weight
        r["dw"] = (gw(x64, w.shape, dy64, padding=1), gw(x64.abs(), w.shape, dy64.abs(), padding=1))
    return r
