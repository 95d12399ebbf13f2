"""GPU parity of the bf16 performance path (tcgen05 GEMM + flash attention) through the C ABI and
the reference-API modules.  Tolerance 2e-2 max-relative (north_star's bf16 bound) against fp32
math on the same bf16-rounded inputs / against the reference-generated golden fixtures."""
import pytest
import torch

from conftest import grad_err, mask_check, relerr
from synth import encoder_data
import adaptersis_b200 as asis
from adaptersis_b200 import kernels as K
from adaptersis_b200._lib import (BF16, EPI_ACCUMULATE, EPI_DGELU, EPI_GELU, EPI_GELU_GRAD, EPI_MUL_AUX, EPI_SCALE_RESIDUAL,
                                  MAJOR_K, MAJOR_MN)

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 2e-2
GEMM_TOL = 2e-3      # fp32 accumulation of exact bf16 products: only summation order differs


@pytest.mark.parametrize("M,N,K_", [(128, 256, 64), (300, 200, 136), (1765, 1024, 1024), (2000, 96, 1024), (70, 32, 40),
                                    (1000, 64, 192), (600, 128, 576), (2000, 48, 320)])      # narrow N: 64- / 128-wide MMAs
@pytest.mark.parametrize("am,bm", [(MAJOR_K, MAJOR_K), (MAJOR_K, MAJOR_MN), (MAJOR_MN, MAJOR_MN), (MAJOR_MN, MAJOR_K)])
def test_gemm_tc_majors(M, N, K_, am, bm):
    torch.manual_seed(0)
    A = torch.randn(M, K_, device=DEV).bfloat16()
    B = torch.randn(N, K_, device=DEV).bfloat16()
    ref = A.float() @ B.float().t()

    def lay(X, major):
        if major == MAJOR_K:
            return X
        Xt = X.t().contiguous()
        if Xt.shape[1] % 8:                       # TMA needs a 16-byte row pitch
            pad = 8 - Xt.shape[1] % 8
            Xt = torch.nn.functional.pad(Xt, (0, pad))[:, :Xt.shape[1] + pad]
        return Xt

    a, b = lay(A, am), lay(B, bm)
    if a.stride(0) % 8 or b.stride(0) % 8:
        with pytest.raises(RuntimeError, match="multiples of 8"):
            K.gemm(BF16, a, am, b, bm, M, N, K_, torch.float32)
        return
    c, _ = K.gemm(BF16, a, am, b, bm, M, N, K_, torch.float32)
    assert relerr(c, ref) < GEMM_TOL


def test_gemm_tc_split_k_weight_gradient():
    for R, N, K_ in ((21180, 1024, 1024),       # ViT-L proj weight gradient: 32 tiles, K = tokens
                     (21168, 96, 1024)):        # a weight gradient of the step with one M tile (1-CTA kernel)
        torch.manual_seed(1)
        dy = torch.randn(R, N, device=DEV).bfloat16()
        x = torch.randn(R, K_, device=DEV).bfloat16()
        ref = dy.float().t() @ x.float()
        dw, _ = K.gemm(BF16, dy, MAJOR_MN, x, MAJOR_MN, N, K_, R, torch.float32)
        assert relerr(dw, ref) < GEMM_TOL
        acc = torch.ones(N, K_, device=DEV)
        dw2, _ = K.gemm(BF16, dy, MAJOR_MN, x, MAJOR_MN, N, K_, R, torch.float32, epilogue=EPI_ACCUMULATE, out=acc)
        assert relerr(dw2, ref + 1) < GEMM_TOL


def test_gemm_tc_epilogues():
    for M, Mt in ((1000, 333), (96, 77)):      # M <= 128: one M tile (1-CTA kernel)
        torch.manual_seed(2)
        N, K_ = 1024, 512
        A = torch.randn(M, K_, device=DEV).bfloat16()
        B = torch.randn(N, K_, device=DEV).bfloat16()
        ref = A.float() @ B.float().t()
        bias = torch.randn(N, device=DEV)
        gamma = torch.randn(N, device=DEV)
        res = torch.randn(M, N, device=DEV)
        c, _ = K.gemm(BF16, A, MAJOR_K, B, MAJOR_K, M, N, K_, torch.bfloat16, bias=bias)
        assert relerr(c.float(), ref + bias) < TOL
        c, aux = K.gemm(BF16, A, MAJOR_K, B, MAJOR_K, M, N, K_, torch.bfloat16, epilogue=EPI_GELU, bias=bias,
                        want_aux_dtype=torch.bfloat16)
        assert relerr(c.float(), torch.nn.functional.gelu(ref + bias)) < TOL and relerr(aux.float(), ref + bias) < TOL
        c, aux = K.gemm(BF16, A, MAJOR_K, B, MAJOR_K, M, N, K_, torch.float32, epilogue=EPI_SCALE_RESIDUAL, bias=bias,
                        gamma=gamma, residual=res, want_aux_dtype=torch.bfloat16)
        assert relerr(c, res + gamma * (ref + bias)) < GEMM_TOL and relerr(aux.float(), ref + bias) < TOL
        h = torch.randn(M, N, device=DEV).bfloat16()
        hh = h.float().requires_grad_(True)
        (dg,) = torch.autograd.grad(torch.nn.functional.gelu(hh), hh, torch.ones_like(hh))
        c, _ = K.gemm(BF16, A, MAJOR_K, B, MAJOR_K, M, N, K_, torch.float32, epilogue=EPI_DGELU, aux=h)
        assert relerr(c, ref * dg) < GEMM_TOL
        # GELU with the derivative saved for the backward, and the backward epilogue that multiplies by it
        pre = (ref + bias).requires_grad_(True)
        (dpre,) = torch.autograd.grad(torch.nn.functional.gelu(pre), pre, torch.ones_like(pre))
        c, aux = K.gemm(BF16, A, MAJOR_K, B, MAJOR_K, M, N, K_, torch.bfloat16, epilogue=EPI_GELU_GRAD, bias=bias,
                        want_aux_dtype=torch.bfloat16)
        assert relerr(c.float(), torch.nn.functional.gelu(ref + bias)) < TOL and relerr(aux.float(), dpre) < TOL
        c, _ = K.gemm(BF16, A, MAJOR_K, B, MAJOR_K, M, N, K_, torch.bfloat16, epilogue=EPI_MUL_AUX, aux=aux)
        assert relerr(c.float(), ref * aux.float()) < TOL
        # the same two on a shape with M / N tails (generic epilogue path)
        Nt = 200
        c, aux = K.gemm(BF16, A[:Mt], MAJOR_K, B[:Nt], MAJOR_K, Mt, Nt, K_, torch.bfloat16, epilogue=EPI_GELU_GRAD, bias=bias[:Nt],
                        want_aux_dtype=torch.bfloat16)
        assert relerr(c.float(), torch.nn.functional.gelu(ref[:Mt, :Nt] + bias[:Nt])) < TOL and relerr(aux.float(), dpre[:Mt, :Nt]) < TOL
        c, _ = K.gemm(BF16, A[:Mt], MAJOR_K, B[:Nt], MAJOR_K, Mt, Nt, K_, torch.float32, epilogue=EPI_MUL_AUX, aux=aux)
        assert relerr(c, ref[:Mt, :Nt] * aux.float()) < GEMM_TOL


@pytest.mark.parametrize("B,T,H", [(1, 128, 1), (2, 300, 3), (1, 1765, 16), (3, 1764, 2)])
def test_attention_tc(B, T, H):
    torch.manual_seed(3)
    C = H * 64
    qkv = torch.randn(B, T, 3 * C, device=DEV).bfloat16()
    x = qkv.float().requires_grad_(True)
    q, k, v = x.view(B, T, 3, H, 64).permute(2, 0, 3, 1, 4)
    s = (q * 64 ** -0.5) @ k.transpose(-1, -2)
    ref = (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(B, T, C)
    dout = torch.randn(B, T, C, device=DEV).bfloat16()
    (g,) = torch.autograd.grad(ref, x, dout.float())
    out, lse = K.attention_forward(BF16, qkv, B, T, H, 64)
    assert relerr(out.float(), ref) < TOL
    assert relerr(lse, torch.logsumexp(s, -1)) < 1e-3
    dqkv = K.attention_backward(BF16, qkv, out, lse, dout, B, T, H, 64)
    for a, b in zip(dqkv.float().view(B, T, 3, C).unbind(2), g.view(B, T, 3, C).unbind(2)):
        assert relerr(a, b) < TOL
    dqkv2 = K.attention_backward(BF16, qkv, out, lse, dout, B, T, H, 64)
    assert torch.equal(dqkv, dqkv2)               # atomic-free: bit-identical run to run


def test_block_bf16_vs_fp32_mode():
    torch.manual_seed(4)
    blk = asis.Block(dim=256, num_heads=4, qkv_bias=True, init_values=1e-5, attn_class=asis.MemEffAttention).to(DEV)
    with torch.no_grad():
        blk.ls1.gamma.normal_(0.5, 0.2)
        blk.ls2.gamma.normal_(0.5, 0.2)
    x = torch.randn(2, 333, 256, device=DEV)
    gy = torch.randn(2, 333, 256, device=DEV)
    res = {}
    for mode in ("fp32", "bf16"):
        with asis.precision(mode):
            xx = x.clone().requires_grad_(True)
            y = blk(xx)
            params = list(blk.parameters())
            res[mode] = (y,) + torch.autograd.grad(y, [xx] + params, gy)
    assert relerr(res["bf16"][0], res["fp32"][0]) < TOL
    assert relerr(res["bf16"][1], res["fp32"][1]) < TOL
    for (name, _), a, b in zip(blk.named_parameters(), res["bf16"][2:], res["fp32"][2:]):
        assert relerr(a, b) < 3e-2, name


def test_composed_encoder_bf16_golden(golden):
    """The bf16 performance mode end to end against the REFERENCE-generated fixture with head_dim 64
    (tcgen05 GEMMs + flash attention + bf16-value MSDA + adapters + decoder + loss, forward and backward).
    Activations and logits: north_star's 2e-2.  Gradients: bf16 rounding through this graph (BatchNorm with batch
    statistics, a very flat dice loss, bilinear-sampling gradients) moves the REFERENCE'S OWN gradients by 4 %
    (median) to 68 % when PyTorch runs it under bf16 autocast -- the fixture stores that per parameter
    (`amp_err`, make_golden.py) -- so every gradient is required to be within max(2e-2, 3 x reference-AMP error).
    Argmax mask: identical wherever the reference's decision is determined at the logits' tolerance."""
    from test_gpu_modules import run_composed
    g = golden("encoder_hd64.pt")
    assert g["cfg"]["dim"] // g["cfg"]["heads"] == 64
    amp = g["amp_err"]
    r = run_composed(g, "bf16")
    e_feat, e_x = grad_err(r["feat"], g["feat"]), grad_err(r["x"], g["x"])
    logits = r["logits"].float()
    e_log = grad_err(logits[:, :, ::4, ::4], g["logits_s4"])
    print(f"[encoder_hd64.pt] bf16 mode: feat {e_feat:.2e} x {e_x:.2e} logits {e_log:.2e} "
          f"(reference under torch bf16 autocast: feat {amp['feat']:.2e} logits {amp['logits']:.2e})")
    assert e_feat < TOL and e_x < TOL
    assert e_log < max(TOL, amp["logits"])
    flips, near = mask_check(logits, g, max(TOL, amp["logits"]))
    print(f"[encoder_hd64.pt] bf16 mode vs reference mask: {flips} flips / {logits[:, 0].numel()} pixels "
          f"({near} near-tie pixels at that tolerance)")
    assert abs(float(r["loss"].detach()) - float(g["loss"])) < max(2e-3, 2 * amp["loss"])
    worst, bad = (0.0, None), []
    for k, gr in r["grads"].items():
        ref = g["grads"][k]
        assert gr is not None, k
        if k not in amp["grads"]:
            continue                      # analytically zero in the reference
        e = grad_err(gr, ref)
        worst = max(worst, (e / max(2e-2, 3 * amp["grads"][k]), k, e))
        if not e < max(2e-2, 3 * amp["grads"][k]):
            bad.append((k, e, amp["grads"][k]))
    print(f"[encoder_hd64.pt] bf16 mode: {len(r['grads'])} gradients, tightest margin at {worst[1]}: error {worst[2]:.2e} "
          f"= {worst[0]:.2f} x its allowance")
    assert not bad, bad[:10]


def test_vit_small_bf16_vs_fp32_taps():
    """ViT-S/14 (head_dim 64), 224x224, batch 2 -- BASELINE.json config 1 backbone: bf16 taps and
    segmentation-style argmax agree with the fp32 parity path."""
    torch.manual_seed(5)
    m = asis.build_model_for_eval("vit_small", img_size=224, patch_size=14).to(DEV)
    with torch.no_grad():
        for blk in m.blocks:
            blk.ls1.gamma.fill_(1.0)
            blk.ls2.gamma.fill_(1.0)
    img = torch.rand(2, 3, 224, 224, device=DEV)
    outs = {}
    for mode in ("fp32", "bf16"):
        with asis.precision(mode), torch.no_grad():
            outs[mode] = m.get_intermediate_layers(img, 4, return_class_token=True)
    for (a, ca), (b, cb) in zip(outs["bf16"], outs["fp32"]):
        assert relerr(a, b) < TOL and relerr(ca, cb) < TOL


def test_attention_run_to_run_identical():
    # the kernels are atomic-free and barrier-ordered: the same input must give the same bits on every
    # launch, also back to back with other kernels (a racy TMEM hand-off once showed up only here)
    B, T, H = 12, 1765, 16
    g = torch.Generator().manual_seed(11)
    qkv = (torch.randn(B, T, 3 * H * 64, generator=g) * 0.5).to(DEV).bfloat16()
    A = torch.randn(B * T, 1024, generator=g).to(DEV).bfloat16()
    W = torch.randn(1024, 1024, generator=g).to(DEV).bfloat16()
    out0, lse0 = K.attention_forward(BF16, qkv, B, T, H, 64)
    dout = torch.randn(out0.shape, generator=g).to(DEV).bfloat16()
    g0 = K.attention_backward(BF16, qkv, out0, lse0, dout, B, T, H, 64)
    assert torch.isfinite(out0.float()).all() and torch.isfinite(lse0).all() and torch.isfinite(g0.float()).all()
    for i in range(30):
        if i % 3 == 0:
            K.gemm(BF16, A, MAJOR_K, W, MAJOR_K, B * T, 1024, 1024, torch.bfloat16)
        out, lse = K.attention_forward(BF16, qkv, B, T, H, 64)
        assert torch.equal(out, out0) and torch.equal(lse, lse0), f"forward differs at repeat {i}"
        if i % 5 == 0:
            assert torch.equal(K.attention_backward(BF16, qkv, out0, lse0, dout, B, T, H, 64), g0), f"backward differs at repeat {i}"


def test_full_size_batch_independence():
    """BASELINE.json's full sizes (ViT-L width, 1765 tokens, 12 images; the injector's MSDA shape): a
    size-independent property the reference has by construction -- every image is processed on its
    own -- checked bit for bit: the 12-image call equals two 6-image calls, for the block's outputs
    and input gradients and for the deformable attention's output and all three gradients."""
    torch.manual_seed(7)
    blk = asis.Block(dim=1024, num_heads=16, qkv_bias=True, init_values=1e-5, attn_class=asis.MemEffAttention).to(DEV)
    with torch.no_grad():
        blk.ls1.gamma.normal_(0.5, 0.2)
        blk.ls2.gamma.normal_(0.5, 0.2)
    x = torch.randn(12, 1765, 1024, device=DEV)
    gy = torch.randn(12, 1765, 1024, device=DEV)
    with asis.precision("bf16"):
        def run(xs, gs):
            xx = xs.clone().requires_grad_(True)
            y = blk(xx)
            (gx,) = torch.autograd.grad(y, xx, gs)
            return y, gx
        y12, g12 = run(x, gy)
        ya, ga = run(x[:6], gy[:6])
        yb, gb = run(x[6:], gy[6:])
    assert torch.isfinite(y12).all() and torch.isfinite(g12).all()
    assert torch.equal(y12, torch.cat([ya, yb])) and torch.equal(g12, torch.cat([ga, gb]))

    shapes = [(73, 73), (36, 36), (18, 18)]
    g = torch.Generator().manual_seed(8)
    S = sum(h * w for h, w in shapes)
    value = torch.randn(12, S, 8, 128, generator=g).to(DEV).bfloat16()
    loc = (torch.rand(12, 1764, 8, 3, 4, 2, generator=g) * 1.1 - 0.05).to(DEV)
    aw = torch.softmax(torch.randn(12, 1764, 8, 12, generator=g), -1).view(12, 1764, 8, 3, 4).to(DEV)
    gout = torch.randn(12, 1764, 1024, generator=g).to(DEV).bfloat16()
    ss = torch.as_tensor(shapes, dtype=torch.long, device=DEV)
    lsi = torch.cat([ss.new_zeros(1), ss.prod(1).cumsum(0)[:-1]])
    o12 = K.msda_forward(value, ss, lsi, loc, aw)
    b12 = K.msda_backward(value, ss, lsi, loc, aw, gout)
    for sl in (slice(0, 6), slice(6, 12)):
        o = K.msda_forward(value[sl], ss, lsi, loc[sl], aw[sl])
        b = K.msda_backward(value[sl], ss, lsi, loc[sl], aw[sl], gout[sl])
        assert torch.equal(o12[sl], o)
        for t12, t in zip(b12, b):
            assert torch.equal(t12[sl], t)
