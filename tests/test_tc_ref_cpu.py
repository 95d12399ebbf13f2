"""The elementwise bounds of tests/tc_ref.py accept what the tensor-core kernels compute and reject results that are
wrong in the ways persistent, tiled kernels go wrong.  No GPU: a host model of each kernel's arithmetic (fp32
accumulation of bf16 products, bf16 P / dS, the forward's lazy rescaling) produces the correct result at small shapes,
and each test then breaks one tile, row group, key block or operand the way an indexing or phase bug would."""
import math

import pytest
import torch

import tc_ref as R

BF = torch.bfloat16
M_, N_, K_ = 256, 512, 256          # 2 x 2 output tiles of 128 x 256, 4 k-blocks of 64


def _bf(t):
    return t.bfloat16().float()


# ------------------------------------------------------------------------------------------------- GEMM
def _gemm_operands(seed=0):
    g = torch.Generator().manual_seed(seed)
    # every M tile and N tile its own scale: a unit that reads another unit's rows is off by O(1)
    A = _bf(torch.randn(M_, K_, generator=g) * (1 + torch.arange(M_) // 128).float()[:, None])
    B = _bf(torch.randn(N_, K_, generator=g) * (1 + 0.5 * (torch.arange(N_) // 256)).float()[:, None])
    return g, A, B


def _gelu32(h):
    return 0.5 * h * (1 + torch.erf(h * 0.5 ** 0.5))


def _dgelu32(h):
    return 0.5 * (1 + torch.erf(h * 0.5 ** 0.5)) + h * torch.exp(-0.5 * h * h) * 0.3989422804014327


def gemm_model(A, B, epilogue, bias=None, gamma=None, residual=None, aux=None, out_dtype=BF, acc=None):
    """The kernel's arithmetic: fp32 accumulation of exact bf16 products, fp32 epilogue, rounding at the store."""
    acc = A @ B.t() if acc is None else acc
    h = acc + (bias if bias is not None else 0.0)
    outs = {}
    if epilogue == "none":
        outs["c"] = h
    elif epilogue == "gelu_grad":
        outs["c"], outs["aux"] = _gelu32(h), _dgelu32(h)
    elif epilogue == "scale_residual":
        outs["c"], outs["aux"] = residual + gamma * h, h
    elif epilogue == "mul_aux":
        outs["c"] = acc * aux
    return {k: (v.to(out_dtype).float() if k == "c" else _bf(v)) for k, v in outs.items()}


def _check_all(outs, refs, out_dtype=BF):
    reps = []
    for name, (ref, terms) in refs.items():
        if name in outs:
            u = R.u_out(out_dtype) if name == "c" else R.U_BF16
            reps.append(R.check(name, outs[name], ref, u, terms, block=(128, 256)))
    return reps


def _accepts(reps):
    for r in reps:
        assert r.ok, str(r)


def _rejects(reps, tile=None):
    bad = [r for r in reps if not r.ok]
    assert bad, "a wrong result passed: " + "; ".join(str(r) for r in reps)
    if tile is not None:      # the report names the broken tile
        assert any(bool(r.slabs[tile] > 1) for r in bad), [str(r) for r in bad]


@pytest.mark.parametrize("out_dtype", [BF, torch.float32])
def test_gemm_bias_chunk_missing(out_dtype):
    g, A, B = _gemm_operands()
    bias = torch.randn(N_, generator=g)
    refs = R.gemm_ref(A, B, "none", bias=bias)
    outs = gemm_model(A, B, "none", bias=bias, out_dtype=out_dtype)
    _accepts(_check_all(outs, refs, out_dtype))
    bad = bias.clone()
    bad[256 + 64:256 + 96] = 0.0                  # one 32-column chunk of tile (1, 1)
    c = gemm_model(A, B, "none", bias=bias, out_dtype=out_dtype, acc=A @ B.t())["c"]
    c[128:256] = gemm_model(A[128:256], B, "none", bias=bad, out_dtype=out_dtype)["c"]
    _rejects(_check_all({"c": c}, refs, out_dtype), tile=(1, 1))


def test_gemm_tile_swapped():
    g, A, B = _gemm_operands(1)
    bias = torch.randn(N_, generator=g)
    refs = R.gemm_ref(A, B, "none", bias=bias)
    c = gemm_model(A, B, "none", bias=bias)["c"]
    c[128:256, 0:256] = c[0:128, 0:256]           # accumulator buffer of the previous tile stored again
    _rejects(_check_all({"c": c}, refs), tile=(1, 0))


def test_gemm_k_block_missing():
    g, A, B = _gemm_operands(2)
    refs = R.gemm_ref(A, B, "none")
    acc = A @ B.t()
    acc[0:128, 256:512] -= A[0:128, 128:192] @ B[256:512, 128:192].t()
    _rejects(_check_all(gemm_model(A, B, "none", acc=acc, out_dtype=torch.float32), refs, torch.float32), tile=(0, 1))


def test_gemm_lane_quarter_shifted():
    g, A, B = _gemm_operands(3)
    refs = R.gemm_ref(A, B, "none")
    c = gemm_model(A, B, "none")["c"]
    c[128 + 32:128 + 64, 256:512] = c[128 + 64:128 + 96, 256:512].clone()     # TMEM lanes 32-63 read from 64-95
    _rejects(_check_all({"c": c}, refs), tile=(1, 1))


def test_gemm_aux_holds_preactivation():
    g, A, B = _gemm_operands(4)
    bias = torch.randn(N_, generator=g)
    refs = R.gemm_ref(A, B, "gelu_grad", bias=bias)
    outs = gemm_model(A, B, "gelu_grad", bias=bias)
    _accepts(_check_all(outs, refs))
    outs["aux"] = _bf(A @ B.t() + bias)           # GELU'(h) expected, h stored
    _rejects(_check_all(outs, refs))


def test_gemm_residual_from_other_tile():
    g, A, B = _gemm_operands(5)
    bias, gamma = torch.randn(N_, generator=g), torch.randn(N_, generator=g)
    res = torch.randn(M_, N_, generator=g) + (torch.arange(M_) // 128).float()[:, None] * 3.0
    refs = R.gemm_ref(A, B, "scale_residual", bias=bias, gamma=gamma, residual=res)
    outs = gemm_model(A, B, "scale_residual", bias=bias, gamma=gamma, residual=res, out_dtype=torch.float32)
    _accepts(_check_all(outs, refs, torch.float32))
    wrong = res.clone()
    wrong[128:256] = res[0:128]                   # the prefetch of the next tile read the previous tile's rows
    outs = gemm_model(A, B, "scale_residual", bias=bias, gamma=gamma, residual=wrong, out_dtype=torch.float32)
    _rejects(_check_all(outs, refs, torch.float32), tile=(1, 0))


def test_gemm_mul_aux_accepts():
    g, A, B = _gemm_operands(6)
    aux = _bf(torch.randn(M_, N_, generator=g))
    refs = R.gemm_ref(A, B, "mul_aux", aux=aux)
    _accepts(_check_all(gemm_model(A, B, "mul_aux", aux=aux), refs))


# -------------------------------------------------------------------------------------------- attention
def attn_forward_model(qkv, H, rescale=True, count_masked_key=False, stale_lse=False):
    """The forward kernel's algorithm in fp32: key tiles of 128, the first tile sets the log2-domain maximum, a later
    tile moves it (and rescales O and l) only when it grows by more than 8, P = ex2(s log2(e) / 8 - m) rounded to bf16
    for P V, l summed from the unrounded exponentials; rows >= T of K / V are TMA's zero fill."""
    Bn, T, _ = qkv.shape
    nkv = (T + 127) // 128
    Tp = nkv * 128
    x = torch.nn.functional.pad(qkv.view(Bn, T, 3, H, 64), (0, 0, 0, 0, 0, 0, 0, Tp - T)).permute(2, 0, 3, 1, 4)
    q, k, v = x[0][:, :, :T], x[1], x[2]
    sl2 = (q @ k.transpose(-1, -2)) * float(R.SCALE * R.LOG2E)
    limit = T + 1 if count_masked_key else T
    sl2[..., limit:] = -math.inf
    O = torch.zeros(Bn, H, T, 64)
    l = torch.zeros(Bn, H, T, 1)
    m = m_first = None
    for j in range(nkv):
        st = sl2[..., j * 128:(j + 1) * 128]
        mx = st.amax(-1, keepdim=True)
        if j == 0:
            m = m_first = mx
        else:
            grow = torch.maximum(m, mx) - m > 8.0
            alpha = torch.where(grow, torch.exp2(m - torch.maximum(m, mx)), torch.ones_like(m))
            m = torch.where(grow, torch.maximum(m, mx), m)
            l = l * alpha
            if rescale:
                O = O * alpha
        p = torch.exp2(st - m)
        l = l + p.sum(-1, keepdim=True)
        O = O + _bf(p) @ v[:, :, j * 128:(j + 1) * 128]
    out = _bf((O / l).permute(0, 2, 1, 3).reshape(Bn, T, H * 64))
    lse = ((m_first if stale_lse else m) + torch.log2(l)).squeeze(-1) * math.log(2)
    return out, lse


def attn_backward_model(qkv, H, out, lse, dout):
    """The backward kernels' arithmetic: P recomputed from lse and rounded to bf16 for dV = P^T dO, dS = P (dP - D)
    rounded to bf16 for dQ and dK, D from the bf16 O, fp32 accumulation."""
    Bn, T, _ = qkv.shape
    x = qkv.view(Bn, T, 3, H, 64).permute(2, 0, 3, 1, 4)
    q, k, v = x[0], x[1], x[2]
    dO = dout.view(Bn, T, H, 64).permute(0, 2, 1, 3)
    O = out.view(Bn, T, H, 64).permute(0, 2, 1, 3)
    P = torch.exp2((q @ k.transpose(-1, -2)) * float(R.SCALE * R.LOG2E) - lse[..., None] * R.LOG2E)
    D = (dO * O).sum(-1, keepdim=True)
    dS = _bf(P * (dO @ v.transpose(-1, -2) - D))
    dV = _bf(P).transpose(-1, -2) @ dO
    dQ = dS @ k * R.SCALE
    dK = dS.transpose(-1, -2) @ q * R.SCALE
    return dQ, dK, dV


def _pack(Bn, T, H, dQ, dK, dV):
    return _bf(torch.stack([dQ, dK, dV], 0).permute(1, 3, 0, 2, 4).reshape(Bn, T, 3 * H * 64))


def _attn_check(qkv, H, out, lse, dqkv=None, dout=None):
    Bn, T = qkv.shape[:2]
    f = R.attention_forward_ref(qkv, H)
    reps = [R.check("out", out, f["out"][0], R.U_BF16, f["out"][1], block=(1, T, 64)),
            R.check("lse", lse, f["lse"][0], 0.0, f["lse"][1], block=(1, 1, T))]
    if dqkv is not None:
        ref, terms = R.attention_backward_ref(qkv, H, dout, f, out)
        reps.append(R.check("dqkv", dqkv, ref, R.U_BF16, terms, block=(1, T, 64)))
    return reps


def _attn_case(kind, Bn=2, T=200, H=2, seed=0):
    g = torch.Generator().manual_seed(seed)
    qkv = R.attention_inputs(kind, Bn, T, H, g)
    dout = _bf(torch.randn(Bn, T, H * 64, generator=g))
    return qkv, dout


@pytest.mark.parametrize("kind,T", [("randn", 200), ("ramp", 300), ("sub", 300), ("qzero", 65), ("ramp", 129)])
def test_attention_model_accepted(kind, T):
    qkv, dout = _attn_case(kind, T=T)
    out, lse = attn_forward_model(qkv, 2)
    dq, dk, dv = attn_backward_model(qkv, 2, out, lse, dout)
    _accepts(_attn_check(qkv, 2, out, lse, _pack(2, T, 2, dq, dk, dv), dout))


def test_attention_inputs_exercise_the_rescale_rule():
    qkv, _ = _attn_case("ramp", T=300)
    fires, margin = R.rescale_sim(qkv, 2)
    n = fires.sum(-1)
    assert int((n >= 2).sum()) > 0 and bool(fires[..., 1].any()) and bool(fires[..., 2].any())
    sub, _ = _attn_case("sub", T=300)
    f2, m2 = R.rescale_sim(sub, 2)
    assert not bool(f2.any()) and float(m2.min()) > 0.3
    q, k, _ = R._split_qkv(sub, 2)
    s = (q @ k.transpose(-1, -2)) * (R.SCALE * R.LOG2E)
    assert float((s.amax(-1) - s[..., :128].amax(-1)).max()) > 7.0      # P reaches > 2^7 without a rescale


def test_attention_rescale_skipped_rejected():
    qkv, _ = _attn_case("ramp", T=300)
    fires, _ = R.rescale_sim(qkv, 2)
    assert bool(fires.any())
    out, lse = attn_forward_model(qkv, 2, rescale=False)
    reps = _attn_check(qkv, 2, out, lse)
    _rejects(reps[:1])
    bad = reps[0].slabs > 1                                             # exactly the (image, head)s where it fires
    assert torch.equal(bad.view(2, 2), fires.any(-1).any(-1))


def test_attention_stale_lse_rejected():
    qkv, _ = _attn_case("ramp", T=300)
    out, lse = attn_forward_model(qkv, 2, stale_lse=True)
    reps = _attn_check(qkv, 2, out, lse)
    assert reps[0].ok
    _rejects(reps[1:])


@pytest.mark.parametrize("T", [65, 100, 200])
def test_attention_masked_key_counted_rejected(T):
    qkv, _ = _attn_case("qzero", T=T)
    out, lse = attn_forward_model(qkv, 2, count_masked_key=True)
    reps = _attn_check(qkv, 2, out, lse)
    assert not reps[0].ok and not reps[1].ok, [str(r) for r in reps]


def test_attention_query_tile_from_other_head_rejected():
    qkv, _ = _attn_case("randn", T=300)
    out, lse = attn_forward_model(qkv, 2)
    o = out.view(2, 300, 2, 64)
    o[1, 128:256, 0] = o[1, 128:256, 1].clone()
    reps = _attn_check(qkv, 2, out, lse)
    _rejects(reps[:1], tile=(1, 0, 0))


def test_attention_dv_last_partial_key_tile_rejected():
    qkv, dout = _attn_case("randn", T=200)
    out, lse = attn_forward_model(qkv, 2)
    dq, dk, dv = attn_backward_model(qkv, 2, out, lse, dout)
    # the last key tile (keys 128..199) misses the contribution of the last, partial query tile
    x = qkv.view(2, 200, 3, 2, 64).permute(2, 0, 3, 1, 4)
    P = torch.exp2((x[0] @ x[1].transpose(-1, -2)) * float(R.SCALE * R.LOG2E) - lse[..., None] * R.LOG2E)
    dO = dout.view(2, 200, 2, 64).permute(0, 2, 1, 3)
    dv = dv.clone()
    dv[:, :, 128:] = _bf(P[:, :, :128, 128:]).transpose(-1, -2) @ dO[:, :, :128]
    reps = _attn_check(qkv, 2, out, lse, _pack(2, 200, 2, dq, dk, dv), dout)
    _rejects(reps[2:])
    assert reps[0].ok and reps[1].ok


def test_conv_reference_matches_unfold():
    """conv3x3_ref against an explicit im2col product (the layout the implicit GEMM uses: K = (ky, kx, cin))."""
    g = torch.Generator().manual_seed(9)
    x = _bf(torch.randn(2, 64, 5, 7, generator=g))
    w = _bf(torch.randn(64, 64, 3, 3, generator=g) * 0.05)
    dy = _bf(torch.randn(2, 64, 5, 7, generator=g))
    r = R.conv3x3_ref(x, w, dy=dy)
    cols = torch.nn.functional.unfold(x.double(), 3, padding=1)                          # [B, Cin*9, HW]
    y = (w.double().view(64, -1) @ cols).view(2, 64, 5, 7)
    assert torch.allclose(r["y"][0], y, rtol=1e-12, atol=1e-12)
    rep = R.check("dw", (torch.einsum("bop,bkp->ok", dy.double().view(2, 64, -1), cols)).view(64, 64, 3, 3),
                  r["dw"][0], R.U_F32, [(R.c_mma(70), r["dw"][1])])
    assert rep.ok, str(rep)
