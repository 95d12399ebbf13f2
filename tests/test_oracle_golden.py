"""Pin the CPU oracle against fixtures produced by the reference's own modules
(tests/golden/make_golden.py).  CPU only.  Tolerance: 2e-5 max-relative in fp32 (pure
re-association noise between two fp32 formulations of the same mathematics)."""
import torch

import pytest

from conftest import as_fixture_entry, grad_err, mask_check, relerr
from synth import adapter_data, encoder_data
import oracle
from oracle import adapter, encoder, layers, masktrans, msda, vit

TOL = 2e-5


def test_msda_core_forward_and_grads(golden):
    for case in golden("msda_core.pt"):
        v = case["value"].clone().requires_grad_(True)
        loc = case["loc"].clone().requires_grad_(True)
        aw = case["aw"].clone().requires_grad_(True)
        out = msda.msda_core(v, case["spatial_shapes"], loc, aw)
        assert relerr(out, case["out"]) < TOL
        gv, gl, ga = torch.autograd.grad(out, (v, loc, aw), case["grad_out"])
        assert relerr(gv, case["grad_value"]) < TOL
        assert relerr(gl, case["grad_loc"]) < TOL
        assert relerr(ga, case["grad_aw"]) < TOL


def test_msda_core_fp64_gradcheck():
    torch.manual_seed(0)
    shapes = [(4, 5), (2, 3)]
    v = torch.randn(1, 26, 2, 4, dtype=torch.double, requires_grad=True)
    loc = (torch.rand(1, 6, 2, 2, 3, 2, dtype=torch.double) * 1.2 - 0.1).requires_grad_(True)
    aw = torch.rand(1, 6, 2, 2, 3, dtype=torch.double, requires_grad=True)
    assert torch.autograd.gradcheck(lambda a, b, c: msda.msda_core(a, shapes, b, c), (v, loc, aw), eps=1e-6, atol=1e-6)


def test_msda_module(golden):
    g = golden("msda_module.pt")
    cfg = g["cfg"]
    kw = dict(n_heads=cfg["n_heads"], n_levels=cfg["n_levels"], n_points=cfg["n_points"])
    out = msda.msda_module(g["sd"], "", g["query"], g["ref"], g["feat"], g["spatial_shapes"], **kw)
    assert relerr(out, g["out"]) < TOL
    out = msda.msda_module(g["sd"], "", g["query"], g["ref"], g["feat"], g["spatial_shapes"], padding_mask=g["mask"], **kw)
    assert relerr(out, g["out_masked"]) < TOL
    out = msda.msda_module(g["sd"], "", g["query"], g["ref4"], g["feat"], g["spatial_shapes"], **kw)
    assert relerr(out, g["out_box"]) < TOL
    assert torch.equal(msda.msda_reset_bias(cfg["n_heads"], cfg["n_levels"], cfg["n_points"]), g["default_bias"])


def test_block(golden):
    g = golden("block.pt")
    sd = {k: v.clone().requires_grad_(True) for k, v in g["sd"].items()}
    x = g["x"].clone().requires_grad_(True)
    nh = g["cfg"]["num_heads"]
    assert relerr(layers.layer_norm(sd, "norm1.", x), g["ln1"]) < TOL
    assert relerr(layers.attention(sd, "attn.", g["ln1"], nh), g["attn"]) < TOL
    y = layers.block(sd, "", x, nh)
    assert relerr(y, g["y"]) < TOL
    names = list(g["grad_params"].keys())
    grads = torch.autograd.grad(y, [x] + [sd[k] for k in names], g["grad_y"])
    assert relerr(grads[0], g["grad_x"]) < TOL
    for k, gr in zip(names, grads[1:]):
        assert relerr(gr, g["grad_params"][k]) < 5e-5, k


def test_vit(golden):
    g = golden("vit.pt")
    cfg = g["cfg"]
    sd = g["sd"]
    assert relerr(vit.patch_embed(sd, "patch_embed.", g["img"], cfg["patch"]), g["patch_tokens"]) < TOL
    assert relerr(vit.interpolate_pos_encoding(sd["pos_embed"], 9, 42, 42, cfg["patch"]), g["pos"]) < TOL
    taps = vit.get_intermediate_layers(sd, g["img"], 4, cfg["num_heads"], cfg["patch"], return_class_token=True)
    assert len(taps) == 4
    for (a, b), (ga, gb) in zip(taps, g["taps"]):
        assert relerr(a, ga) < TOL and relerr(b, gb) < TOL
    nn_ = vit.get_intermediate_layers(sd, g["img"], [1, 3], cfg["num_heads"], cfg["patch"], norm=False, reshape=True)
    for a, ga in zip(nn_, g["taps_nonorm"]):
        assert a.shape == ga.shape and relerr(a, ga) < TOL
    assert relerr(taps[-1][1], g["x_norm_clstoken"]) < TOL


def test_adapter_blocks(golden):
    g = golden("adapter.pt")
    dim = g["cfg"]["dim"]
    x, c, gx, gc = adapter_data(dim)
    assert abs(float(x.double().sum() - g["x_sum"])) < 1e-6 and abs(float(c.double().sum() - g["c_sum"])) < 1e-6
    d1, d2 = adapter.deform_inputs(588, 588, 14)
    for a, b in zip(d1 + d2, g["d1"] + g["d2"]):
        assert a.shape == b.shape and torch.equal(a, b)
    inj = {k: v.clone().requires_grad_(True) for k, v in g["inj_sd"].items()}
    ext = {k: v.clone().requires_grad_(True) for k, v in g["ext_sd"].items()}
    # F4: with the constructor's gamma == 0 the injector is a bit-exact identity
    zero = dict(g["inj_sd"]); zero["gamma"] = torch.zeros(dim)
    assert torch.equal(adapter.cavit(zero, "", x[:, :64], d1[0][:, :64], c, d1[1], n_levels=3), x[:, :64])
    xg = x.clone().requires_grad_(True)
    cg = c.clone().requires_grad_(True)
    x1 = adapter.cavit(inj, "", xg, d1[0], cg, d1[1], n_levels=3)
    c1 = adapter.cacnn(ext, "", cg, d2[0], x1, d2[1], 36, 36, n_levels=1)
    assert relerr(x1, g["x1"]) < TOL
    assert grad_err(c1, g["c1"]) < TOL
    ni, ne = list(g["grad_inj"]), list(g["grad_ext"])
    grads = torch.autograd.grad([x1, c1], [xg, cg] + [inj[k] for k in ni] + [ext[k] for k in ne], [gx, gc])
    assert relerr(grads[0], g["grad_x"]) < TOL
    assert grad_err(grads[1], g["grad_c"]) < TOL
    for k, gr in zip(ni, grads[2:2 + len(ni)]):
        assert relerr(gr, g["grad_inj"][k]) < 1e-4, k
    for k, gr in zip(ne, grads[2 + len(ni):]):
        assert relerr(gr, g["grad_ext"][k]) < 1e-4, k


def _oracle_step(g, dtype):
    """The composed train.py data flow through the oracle in `dtype`: internals + gradients of loss + aux."""
    cfg = g["cfg"]
    img, target, gfeat = encoder_data(1, 588, 3 * cfg["dim"], 42)
    sds = {}
    for tag in ("vit", "spm", "inj", "ext", "dec"):
        sds[tag] = {k: (v.to(dtype).requires_grad_(True) if v.is_floating_point() else v) for k, v in g[tag + "_sd"].items()}
    res = encoder.adapter_encoder(sds["vit"], sds["spm"], sds["inj"], sds["ext"], img.to(dtype), cfg["heads"])
    feat = res["feat"]
    logits = encoder.feature_decoder(sds["dec"], feat)
    logits = torch.nn.functional.interpolate(logits, size=(588, 588), mode="bilinear")
    loss = encoder.dice_loss(torch.softmax(logits, 1), target)
    aux = (feat * gfeat.to(dtype)).sum() / feat.numel() ** 0.5
    names, params = [], []
    for key in g["grads"]:
        tag, k = key.split(".", 1)
        names.append(key)
        params.append(sds[tag][k])
    grads = torch.autograd.grad(loss + aux, params, allow_unused=True)
    return dict(feat=feat.detach(), x=res["x"].detach(), logits=logits.detach(), loss=loss.detach(), aux=aux.detach(),
                grads=dict(zip(names, grads)), img=img, target=target)


@pytest.mark.parametrize("fixture", ["encoder.pt", "encoder_hd64.pt"])
def test_composed_encoder(golden, fixture):
    g = golden(fixture)
    o = _oracle_step(g, torch.float32)
    assert torch.equal(o["img"][:, :, ::28, ::28], g["img_lowres"])
    assert int(o["target"].sum()) == g["target_sum"]
    assert grad_err(o["feat"], g["feat"]) < 5e-5
    assert grad_err(o["x"], g["x"]) < 5e-5
    logits = o["logits"]
    assert relerr(logits[:, :, ::12, ::12], g["logits_lowres"]) < 1e-4
    assert grad_err(logits[:, :, ::4, ::4], g["logits_s4"]) < 1e-4
    # the reference's argmax segmentation mask, every pixel (not a checksum): identical wherever the decision is
    # numerically determined; flips are only tolerated at near-ties (margin < 1e-4 max|logit|) and counted
    flips, near = mask_check(logits, g, 1e-4)
    print(f"[{fixture}] oracle fp32 vs reference mask: {flips} flips / {logits[:, 0].numel()} pixels ({near} near-ties)")
    assert flips <= 3
    assert abs(float(o["loss"] - g["loss"])) < 1e-6
    assert abs(float(o["aux"] - g["aux"])) < 1e-4 * max(1.0, abs(float(g["aux"])))
    checked = 0
    for key, gr in o["grads"].items():
        ref = g["grads"][key]
        assert gr is not None, key
        if not isinstance(ref, dict) and float(ref.abs().max()) < 1e-7:
            # analytically zero (a conv bias in front of a BatchNorm): both sides are rounding noise
            assert float(gr.abs().max()) < 1e-7, key
        else:
            assert grad_err(gr, ref) < 2e-3, key
        checked += 1
    assert checked > 100


@pytest.mark.parametrize("fixture", ["encoder.pt", "encoder_hd64.pt"])
def test_gradient_tolerance_is_fp32_summation_noise(golden, fixture):
    """Why parameter gradients are held to 2e-3 and not 1e-4: measure the REFERENCE's own fp32 gradients (the
    fixture) and the fp32 oracle against an fp64 evaluation of the same graph.  Both sit at the same distance
    from the fp64 truth -- the tolerance is the fp32 summation-order noise of 1e4..1e6-term sums, present in the
    reference itself, not slack for the implementation."""
    g = golden(fixture)
    o64 = _oracle_step(g, torch.float64)
    o32 = _oracle_step(g, torch.float32)
    worst_ref = worst_o32 = 0.0
    table = []
    for key, g64 in o64["grads"].items():
        ref = g["grads"][key]
        if g64 is None or float(g64.abs().max()) < 1e-7:
            continue
        e_ref = grad_err(g64, ref)                    # reference fp32 vs fp64 truth (normalised by the reference's max)
        e_o32 = relerr(o32["grads"][key], g64)
        worst_ref, worst_o32 = max(worst_ref, e_ref), max(worst_o32, e_o32)
        table.append((e_ref, e_o32, key))
        # the fp32 oracle is never further from the truth than a few times the reference itself (+ a 2e-3 floor:
        # the oracle's composite BatchNorm is a little less accurate in fp32 than ATen's fused one, which accumulates in double on the CPU)
        assert e_o32 < max(2e-3, 6 * e_ref), (key, e_o32, e_ref)
    print(f"[{fixture}] worst fp32-vs-fp64 gradient error: reference {worst_ref:.2e}, oracle fp32 {worst_o32:.2e}")
    for e_ref, e_o32, key in sorted(table, reverse=True)[:5]:
        print(f"    {key}: reference {e_ref:.2e}  oracle fp32 {e_o32:.2e}")
    assert worst_ref < 1e-2 and worst_o32 < 1e-2
    # activations: fp32 is within 1e-4 of fp64, and so is the fixture
    assert grad_err(o64["feat"], g["feat"]) < 1e-4 and relerr(o32["feat"], o64["feat"]) < 1e-4
    assert grad_err(o64["logits"][:, :, ::4, ::4], g["logits_s4"]) < 1e-4


def test_mask_transformer(golden):
    # BASELINE config[3]'s decoder: the oracle vs the reference's own MaskTransformer (eval mode), logits, resized logits,
    # arg-max prediction bit for bit, and every gradient
    g = golden("masktrans.pt")
    c = g["cfg"]
    sd = {k: v.clone().requires_grad_(True) for k, v in g["sd"].items()}
    x = g["x"].clone().requires_grad_(True)
    im = (c["gs"] * 14, c["gs"] * 14)
    masks = masktrans.mask_transformer(sd, x, im, 14, c["n_cls"], c["heads"])
    assert masks.shape == g["masks"].shape and relerr(masks, g["masks"]) < TOL
    out, pred = masktrans.segment(masks.detach(), im)
    assert relerr(out, g["logits"]) < TOL
    assert torch.equal(pred.to(torch.uint8), g["pred"])
    names = [n for n in g["grads"] if n != "input"]
    grads = torch.autograd.grad(masks, [x] + [sd[n] for n in names], g["gy"])
    for n, a in zip(["input"] + names, grads):
        assert grad_err(a, g["grads"][n]) < 5 * TOL, n


def test_oracle_is_test_infrastructure_only():
    """No file under the product package may import the oracle."""
    import os
    import re
    root = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "adaptersis_b200")
    bad = []
    for dp, _, fs in os.walk(root):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                src = open(os.path.join(dp, f)).read()
                if re.search(r"^\s*(from|import)\s+oracle\b", src, re.M):
                    bad.append(os.path.join(dp, f))
    assert not bad, bad
    assert "TEST INFRASTRUCTURE ONLY" in oracle.__doc__
