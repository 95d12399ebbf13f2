"""Accuracy of the persistent tensor-core kernels past their first work unit, against fp64 with elementwise bounds
(tests/tc_ref.py).  Every case runs under torch.profiler and asserts from the trace which kernel instantiation ran
and that its grid is smaller than its unit count (the launcher's arithmetic, with the device's SM count), so the
barrier phases, TMEM double buffers and prefetches that only run from a CTA's second unit on are covered.  Operands
carry a scale or offset per M tile / (image, head), so a unit that reads another unit's data fails in its own slab.
Each case prints the kernel, its units per CTA (cluster for the pair kernel), the rescale counts and the largest
err / bound ratio."""
import math
import time

import pytest
import torch

import tc_ref as R
from adaptersis_b200 import kernels as K
from adaptersis_b200._lib import (BF16, EPI_ACCUMULATE, EPI_DGELU, EPI_GELU, EPI_GELU_GRAD, EPI_MUL_AUX, EPI_NONE,
                                  EPI_SCALE_RESIDUAL, MAJOR_K, MAJOR_MN)

pytestmark = pytest.mark.gpu
DEV = "cuda"
BF, F32 = torch.bfloat16, torch.float32


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------------------------------------- GEMM
def gemm_launch(M, N, K_, out_f32, epi, has_bias):
    """gemm_tc_launch's arithmetic: tiles, split-K, clusters (1-CTA kernel when M <= 128)."""
    m_tiles, n_tiles, kb = -(-M // 128), -(-N // 256), -(-K_ // 64)
    CL = 1 if m_tiles == 1 else 2
    m_groups = -(-m_tiles // CL)
    tiles = m_groups * CL * n_tiles
    n = sms()
    splits = 1
    if out_f32 and (epi == EPI_ACCUMULATE or (epi == EPI_NONE and not has_bias)) and tiles * 2 <= n and kb >= 16:
        splits = max(1, min(n // tiles, kb // 8))
    kps = -(-kb // splits)
    splits = -(-kb // kps)
    units = m_groups * n_tiles * splits
    clusters = min(units, n // CL)
    return dict(grid=clusters * CL, units=units, clusters=clusters, splits=splits)


EPI_NAME = {EPI_NONE: "none", EPI_GELU: "gelu", EPI_SCALE_RESIDUAL: "scale_residual", EPI_DGELU: "dgelu",
            EPI_GELU_GRAD: "gelu_grad", EPI_MUL_AUX: "mul_aux", EPI_ACCUMULATE: "accumulate"}
KM = {MAJOR_K: "K", MAJOR_MN: "MN"}

# (name, M, N, K, a_major, b_major, epilogue, out dtype, bias, aux: None / "out" (saved) / "in", kernel)
R_STEP = 21180              # tokens of the training step (12 x 1765)
GEMM_CASES = [
    ("qkv", R_STEP, 3072, 1024, MAJOR_K, MAJOR_K, EPI_NONE, BF, True, None, "gemm_tc_pair_kernel<0, 0, 0, 1, -1>"),
    ("proj f32", R_STEP, 1024, 1024, MAJOR_K, MAJOR_K, EPI_NONE, F32, True, None, "gemm_tc_pair_kernel<0, 0, 0, 0, -1>"),
    ("fc1 gelu lean", R_STEP, 4096, 1024, MAJOR_K, MAJOR_K, EPI_GELU, BF, True, None, "gemm_tc_pair_kernel<0, 0, 1, 1, -1>"),
    ("proj +res aux", R_STEP, 1024, 1024, MAJOR_K, MAJOR_K, EPI_SCALE_RESIDUAL, F32, True, "out", "gemm_tc_pair_kernel<0, 0, 2, 0, 1>"),
    ("fc2 +res", R_STEP, 1024, 4096, MAJOR_K, MAJOR_K, EPI_SCALE_RESIDUAL, F32, True, None, "gemm_tc_pair_kernel<0, 0, 2, 0, 0>"),
    ("fc1 gelu_grad", R_STEP, 4096, 1024, MAJOR_K, MAJOR_K, EPI_GELU_GRAD, BF, True, "out", "gemm_tc_pair_kernel<0, 0, 5, 1, -1>"),
    ("qkv dgrad", R_STEP, 1024, 3072, MAJOR_K, MAJOR_MN, EPI_NONE, BF, False, None, "gemm_tc_pair_kernel<0, 1, 0, 1, -1>"),
    ("fc1 dgrad x gelu'", R_STEP, 1024, 4096, MAJOR_K, MAJOR_MN, EPI_MUL_AUX, BF, False, "in", "gemm_tc_pair_kernel<0, 1, 6, 1, -1>"),
    ("wgrad f32", 4096, 4096, 2048, MAJOR_MN, MAJOR_MN, EPI_NONE, F32, False, None, "gemm_tc_pair_kernel<1, 1, 0, 0, -1>"),
    ("generic K/K dgelu", R_STEP, 1024, 1024, MAJOR_K, MAJOR_K, EPI_DGELU, F32, False, "in", "gemm_tc_pair_kernel<0, 0, -1, -1, -1>"),
    ("generic K/MN f32", R_STEP, 1024, 1024, MAJOR_K, MAJOR_MN, EPI_NONE, F32, False, None, "gemm_tc_pair_kernel<0, 1, -1, -1, -1>"),
    ("generic MN/MN bf16", 4096, 3072, 2048, MAJOR_MN, MAJOR_MN, EPI_NONE, BF, True, None, "gemm_tc_pair_kernel<1, 1, -1, -1, -1>"),
    ("generic MN/K accumulate", R_STEP, 1024, 1024, MAJOR_MN, MAJOR_K, EPI_ACCUMULATE, F32, False, None, "gemm_tc_pair_kernel<1, 0, -1, -1, -1>"),
]


def _tail(M, N, K_):
    """odd m_tiles, N not a multiple of 256 (lean and generic slabs in one launch), K % 64 != 0; pitches stay 16-byte."""
    mt = -(-M // 128)
    if mt % 2 == 0:
        M = (mt - 1) * 128 - 8
    return M, N - 24, K_ - 24


def _lay(X, major):
    """X [rows, K] in the operand's major: MN-major is X^T, its row pitch padded to a multiple of 8 (TMA's 16 bytes)
    when the rows are not (M = 21180 tokens); the kernel reads the first `rows` columns."""
    if major == MAJOR_K:
        return X
    Xt = X.t().contiguous()
    if Xt.shape[1] % 8:
        Xt = torch.nn.functional.pad(Xt, (0, 8 - Xt.shape[1] % 8))
    return Xt


def run_gemm_case(name, M, N, K_, am, bm, epi, odt, has_bias, aux_mode, kern, ldc_pad=0, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    rows = lambda n, blk: (1 + (torch.arange(n, device=DEV) // blk) % 5).float()[:, None] * 0.5   # per-tile scale
    A = (torch.randn(M, K_, device=DEV, generator=g) * rows(M, 128)).bfloat16()
    B = (torch.randn(N, K_, device=DEV, generator=g) * rows(N, 256)).bfloat16()
    bias = torch.randn(N, device=DEV, generator=g) if has_bias else None
    gamma = torch.randn(N, device=DEV, generator=g) if epi == EPI_SCALE_RESIDUAL else None
    ldc = N + ldc_pad
    out_full = torch.empty(M, ldc, dtype=odt, device=DEV)
    out = out_full[:, :N]
    res = c_old = aux_in = None
    kw = {}
    if epi == EPI_SCALE_RESIDUAL:
        res_full = torch.randn(M, ldc, device=DEV, generator=g) + rows(M, 128) * 4
        res = res_full[:, :N]                          # the residual is read with C's row pitch
        kw["residual"] = res
    if epi == EPI_ACCUMULATE:
        out.copy_(torch.randn(M, N, device=DEV, generator=g) + rows(M, 128))
        c_old = out.clone()
    if aux_mode == "in":
        aux_in = (torch.randn(M, N, device=DEV, generator=g) * (1.5 if epi == EPI_DGELU else 1.0)).bfloat16()
        kw["aux"] = aux_in
    if aux_mode == "out":
        kw["want_aux_dtype"] = BF
    a, b = _lay(A, am), _lay(B, bm)
    launch = gemm_launch(M, N, K_, odt == F32, epi, has_bias)
    t0 = time.time()
    (c, aux), ks = R.traced(lambda: K.gemm(BF16, a, am, b, bm, M, N, K_, odt, epilogue=epi, bias=bias, gamma=gamma, out=out,
                                         **kw))
    kname = R.expect_kernel(ks, kern, (launch["grid"],))
    refs = R.gemm_ref(A, B, EPI_NAME[epi], bias=bias, gamma=gamma, residual=res, aux=aux_in, c_old=c_old,
                      splits=launch["splits"])
    reps = [R.check("c", c, refs["c"][0], R.u_out(odt), refs["c"][1], block=(128, 256))]
    if aux is not None and "aux" in refs:
        reps.append(R.check("aux", aux, refs["aux"][0], R.U_BF16, refs["aux"][1], block=(128, 256)))
    upc = launch["units"] / launch["clusters"]
    worst = max(reps, key=lambda r: r.ratio)
    print(f"[gemm {name}] M={M} N={N} K={K_} {KM[am]}/{KM[bm]} ldc={ldc} {kname.split('(')[0]}: grid {launch['grid']}, "
          f"{launch['units']} units = {upc:.2f} per {'cluster' if launch['grid'] != launch['clusters'] else 'CTA'}; "
          f"max err/bound {worst.ratio:.3g} ({worst.name}) [{time.time() - t0:.1f} s]")
    for r in reps:
        assert r.ok, str(r)
    return launch


@pytest.mark.parametrize("tail", [False, True], ids=["step", "tail"])
@pytest.mark.parametrize("case", GEMM_CASES, ids=[c[0] for c in GEMM_CASES])
def test_gemm_persistent(case, tail):
    name, M, N, K_, am, bm, epi, odt, has_bias, aux_mode, kern = case
    if tail:
        M, N, K_ = _tail(M, N, K_)
    launch = run_gemm_case(name + (" tail" if tail else ""), M, N, K_, am, bm, epi, odt, has_bias, aux_mode, kern)
    assert launch["units"] >= 2 * launch["clusters"] and launch["units"] % launch["clusters"], launch   # ragged last wave


# one strided-output case per epilogue family: C (and the residual) as column slices of a wider matrix, ldc != N
STRIDED = [("none", EPI_NONE, BF, True, None, MAJOR_K, "gemm_tc_pair_kernel<0, 0, 0, 1, -1>"),
           ("gelu", EPI_GELU, BF, True, None, MAJOR_K, "gemm_tc_pair_kernel<0, 0, 1, 1, -1>"),
           ("scale_residual", EPI_SCALE_RESIDUAL, F32, True, "out", MAJOR_K, "gemm_tc_pair_kernel<0, 0, 2, 0, 1>"),
           ("gelu_grad", EPI_GELU_GRAD, BF, True, "out", MAJOR_K, "gemm_tc_pair_kernel<0, 0, 5, 1, -1>"),
           ("mul_aux", EPI_MUL_AUX, BF, False, "in", MAJOR_MN, "gemm_tc_pair_kernel<0, 1, 6, 1, -1>"),
           ("dgelu", EPI_DGELU, F32, False, "in", MAJOR_K, "gemm_tc_pair_kernel<0, 0, -1, -1, -1>"),
           ("accumulate", EPI_ACCUMULATE, F32, False, None, MAJOR_K, "gemm_tc_pair_kernel<0, 0, -1, -1, -1>")]


@pytest.mark.parametrize("case", STRIDED, ids=[c[0] for c in STRIDED])
def test_gemm_strided_output(case):
    fam, epi, odt, has_bias, aux_mode, bm, kern = case
    run_gemm_case(f"{fam} ldc != N", 4000, 1000, 512, MAJOR_K, bm, epi, odt, has_bias, aux_mode, kern, ldc_pad=72, seed=1)


def test_gemm_single_cta_kernel_many_n_tiles():
    """M <= 128 runs the 1-CTA kernel over the N tiles; more than one wave of them (bf16 out: no split-K)."""
    N = sms() * 256 + 700
    launch = run_gemm_case("1-CTA", 100, N, 200, MAJOR_K, MAJOR_K, EPI_NONE, BF, True, None, "gemm_tc_kernel<0, 0>", seed=2)
    assert launch["units"] > launch["grid"]


# -------------------------------------------------------------------------------------------- attention
ATTN_CASES = ([(12, 1765, 16, kind) for kind in ("randn", "ramp", "sub", "qzero")] +
              [(12, 1765, 12, "ramp"), (3, 1537, 16, "randn"), (3, 1537, 16, "ramp"), (40, 129, 8, "ramp"),
               (40, 129, 8, "qzero")] +
              [(2, T, 3, kind) for T in (1, 63, 64, 65, 127, 128, 191, 255, 257) for kind in ("ramp", "qzero")])


def _rescale_stats(fires, Bn, T, H, grid, npair):
    """where the host simulation fires: rows, events, tile 1, rows with >= 2, the masked last tile, the second query
    tile of a pair, and a CTA's second or later item."""
    nkv = fires.shape[-1]
    t = torch.arange(T, device=fires.device)
    pr = (t // 128) // 2
    item = (torch.arange(Bn, device=fires.device)[:, None, None] * H + torch.arange(H, device=fires.device)[None, :, None]) * npair + pr
    later = (item // grid) >= 1                                                        # [B, H, T]
    row_any = fires.any(-1)
    return dict(rows=int(row_any.sum()), events=int(fires.sum()), tile1=int(fires[..., 1].sum()) if nkv > 1 else 0,
                multi=int((fires.sum(-1) >= 2).sum()),
                masked_last=int(fires[..., -1].sum()) if (T % 128 and nkv > 1) else 0,
                pair_second=int((row_any & ((t // 128) % 2 == 1)).sum()),
                later_item=int((row_any & later).sum()))


@pytest.mark.parametrize("Bn,T,H,kind", ATTN_CASES, ids=[f"{b}x{t}x{h}-{k}" for b, t, h, k in ATTN_CASES])
def test_attention_persistent(Bn, T, H, kind):
    t0 = time.time()
    g = torch.Generator().manual_seed(Bn * 100003 + T * 31 + H)
    qkv = R.attention_inputs(kind, Bn, T, H, g).to(DEV).bfloat16()
    dout = torch.randn(Bn, T, H * 64, generator=g).to(DEV).bfloat16()
    items, grid, npair = R.attn_units(Bn, T, H, sms())
    (out, lse), ks = R.traced(lambda: K.attention_forward(BF16, qkv, Bn, T, H, 64))
    kf = R.expect_kernel(ks, "attn_fwd8_kernel", (grid,))
    dqkv, ks = R.traced(lambda: K.attention_backward(BF16, qkv, out, lse, dout, Bn, T, H, 64))
    nqb = -(-T // 128)
    R.expect_kernel(ks, "attn_bwd_dkdv_kernel", (nqb, H, Bn))
    R.expect_kernel(ks, "attn_bwd_dq_kernel", (nqb, H, Bn))
    if items >= 2 * sms():
        assert grid < items

    worst = {}
    fires_all = []
    for b in range(Bn):                              # the fp64 reference, one image at a time
        x = qkv[b:b + 1].float()
        f = R.attention_forward_ref(x, H)
        reps = [R.check("out", out[b:b + 1], f["out"][0], R.U_BF16, f["out"][1], block=(1, T, 64)),
                R.check("lse", lse[b:b + 1], f["lse"][0], 0.0, f["lse"][1], block=(1, 1, T))]
        ref, terms = R.attention_backward_ref(x, H, dout[b:b + 1].float(), f, out[b:b + 1])
        reps.append(R.check("dqkv", dqkv[b:b + 1], ref, R.U_BF16, terms, block=(1, T, 64)))
        for r in reps:
            assert r.ok, f"image {b}: {r}"
            if r.ratio >= worst.get(r.name, (-1.0,))[0]:
                worst[r.name] = (r.ratio, b)
        fires, margin = R.rescale_sim(x, H)
        fires_all.append(fires)
        # known answers: a one-key-dominant row is v_k, a q = 0 row is the mean of V
        P = f["_P"]
        q0 = (f["_q"] == 0).all(-1)                                                   # [1, H, T]
        o = out[b:b + 1].double().view(1, T, H, 64).permute(0, 2, 1, 3)
        v = f["_v"]
        if bool(q0.any()):
            e = (o - v.mean(-2, keepdim=True)).abs()[q0]
            assert bool((e <= R.U_BF16 * v.abs().amax(-2, keepdim=True).expand_as(o)[q0] + 1e-6).all())
        dom = P.amax(-1) > 1 - 2.0 ** -20
        if bool(dom.any()):
            vk = torch.gather(v, 2, P.argmax(-1, keepdim=True).expand(-1, -1, -1, 64))
            assert bool(((o - vk).abs()[dom] <= 2 * R.U_BF16 * vk.abs()[dom] + 2.0 ** -19 * float(v.abs().max())).all())
        del f, ref, terms, P
    fires = torch.cat(fires_all)
    st = _rescale_stats(fires, Bn, T, H, grid, npair)
    print(f"[attention {Bn}x{T}x{H} {kind}] {kf.split('(')[0]}: {items} items on grid {grid} = "
          f"{items / grid:.2f} per CTA; rescale fires {st}; max err/bound "
          + ", ".join(f"{k} {v[0]:.3g} (image {v[1]})" for k, v in worst.items()) + f" [{time.time() - t0:.1f} s]")
    nkv = -(-T // 128)
    if kind == "ramp":
        if nkv >= 2:
            assert st["tile1"] > 0 and (T % 128 == 0 or st["masked_last"] > 0)
        if nkv >= 3:
            assert st["multi"] > 0
        if nqb >= 2:
            assert st["pair_second"] > 0
        if items > grid and nkv >= 2:
            assert st["later_item"] > 0
    if kind == "sub":
        assert st["events"] == 0


# ----------------------------------------------------------------------------------------- convolution
CONV_CASES = [(4, 100, 100, 64, 64), (2, 40, 40, 128, 128), (1, 40, 40, 64, 256)]


def conv_launch(op, Bn, H, W, Cin, Cout):
    Rr = Bn * (H + 2) * (W + 2)
    n = sms()
    if op == 2:
        m_groups, n_tiles, kb = (-(-Cout // 128) + 1) // 2, -(-9 * Cin // 256), -(-Rr // 64)
        tiles = m_groups * n_tiles
        splits = max(1, min((n // 2) // tiles, kb // 8, 64))
        kps = -(-kb // splits)
        splits = -(-kb // kps)
        units = tiles * splits
    else:
        m_groups, n_tiles, splits = (-(-Rr // 128) + 1) // 2, -(-(Cout if op == 0 else Cin) // 256), 1
        units, kps = m_groups * n_tiles, 9 * (Cin if op == 0 else Cout) // 64
    clusters = min(units, n // 2)
    return dict(grid=2 * clusters, units=units, clusters=clusters, splits=splits, k=kps * 64)


@pytest.mark.parametrize("Bn,H,W,Cin,Cout", CONV_CASES)
def test_conv3x3_persistent(Bn, H, W, Cin, Cout):
    t0 = time.time()
    F = torch.nn.functional
    g = torch.Generator().manual_seed(H * 7 + Cout)
    img = (1 + torch.arange(Bn)).float().view(Bn, 1, 1, 1) * 0.5                        # per-image scale
    x = (torch.randn(Bn, Cin, H, W, generator=g) * img).bfloat16().to(DEV)
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) * 0.05).bfloat16().to(DEV)
    bias = torch.randn(Cout, generator=g).to(DEV)
    dy = (torch.randn(Bn, Cout, H, W, generator=g) * img).bfloat16().to(DEV)
    nhwc_pad = lambda t: F.pad(t.permute(0, 2, 3, 1), (0, 0, 1, 1, 1, 1)).contiguous()
    xp, dyp = nhwc_pad(x), nhwc_pad(dy)
    w2 = w.permute(0, 2, 3, 1).reshape(Cout, 9 * Cin).contiguous()
    yp = torch.empty(Bn, H + 2, W + 2, Cout, dtype=BF, device=DEV)
    dxp = torch.empty_like(xp)
    dw2 = torch.empty(Cout, 9 * Cin, dtype=F32, device=DEV)
    refs = R.conv3x3_ref(x, w, bias, dy)
    inner = lambda t: t[:, 1:-1, 1:-1].permute(0, 3, 1, 2)
    outs = [("y", 0, lambda: K.conv3x3s1_gemm(0, xp, w2, yp, bias, Bn, H, W, Cin, Cout), lambda: inner(yp),
             "gemm_tc_pair_kernel<0, 0, 0, 1, -1>", R.U_BF16),
            ("dx", 1, lambda: K.conv3x3s1_gemm(1, dyp, w2, dxp, None, Bn, H, W, Cin, Cout), lambda: inner(dxp),
             "gemm_tc_pair_kernel<0, 1, 0, 1, -1>", R.U_BF16),
            ("dw", 2, lambda: K.conv3x3s1_gemm(2, dyp, xp, dw2, None, Bn, H, W, Cin, Cout),
             lambda: dw2.view(Cout, 3, 3, Cin).permute(0, 3, 1, 2), "gemm_tc_pair_kernel<1, 1, 0, 0, -1>", R.U_F32)]
    msg = []
    for name, op, run, view, kern, u in outs:
        launch = conv_launch(op, Bn, H, W, Cin, Cout)
        _, ks = R.traced(run)
        R.expect_kernel(ks, kern, (launch["grid"],))
        ref, sh = refs[name]
        c = R.c_mma(launch["k"], launch["splits"]) + (R.C_EPI if op == 0 else 0.0)
        rep = R.check(name, view(), ref, u, [(c, sh)])
        assert rep.ok, f"op {op}: {rep}"
        msg.append(f"op {op} {kern}: {launch['units']} units / {launch['clusters']} clusters = "
                   f"{launch['units'] / launch['clusters']:.2f}, max err/bound {rep.ratio:.3g}")
        if op == 0 and (Bn, H, W) == (4, 100, 100):
            assert launch["units"] >= 2 * launch["clusters"]
    print(f"[conv3x3 B={Bn} {H}x{W} {Cin}->{Cout}] " + "; ".join(msg) + f" [{time.time() - t0:.1f} s]")
