"""GPU parity of the reference-API modules in fp32 parity mode against the reference-generated
golden fixtures (outputs AND gradients): Block, DinoVisionTransformer, CAViT/CACNN, and the
composed adapter encoder + decoder + loss of train.py.  Tolerance: 1e-4 max-relative on
activations / logits, argmax masks bit-exact; parameter gradients 2e-3 of their own max (they
are sums over ~1e4-1e6 fp32 terms in a different order than the reference's)."""
import pytest
import torch

from conftest import grad_err, mask_check, relerr
from synth import adapter_data, encoder_data
import adaptersis_b200 as asis
from oracle import encoder as o_enc

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-4
GTOL = 2e-3


def test_block_golden(golden):
    g = golden("block.pt")
    blk = asis.Block(dim=64, num_heads=4, mlp_ratio=4.0, qkv_bias=True, proj_bias=True, ffn_bias=True, init_values=1e-5,
                     attn_class=asis.MemEffAttention).to(DEV)
    blk.load_state_dict(g["sd"])
    with asis.precision("fp32"):
        x = g["x"].to(DEV).requires_grad_(True)
        y = blk(x)
        assert relerr(y, g["y"]) < TOL
        names = list(g["grad_params"])
        params = dict(blk.named_parameters())
        grads = torch.autograd.grad(y, [x] + [params[k] for k in names], g["grad_y"].to(DEV))
        assert relerr(grads[0], g["grad_x"]) < TOL
        for k, gr in zip(names, grads[1:]):
            assert relerr(gr, g["grad_params"][k]) < 5e-4, k
        # stand-alone sub-modules keep working too (reference API)
        assert relerr(blk.attn(g["ln1"].to(DEV)), g["attn"]) < TOL
        xd = g["x"].to(DEV)
        mlp_in = torch.nn.functional.layer_norm(xd + blk.ls1(blk.attn(g["ln1"].to(DEV))), (64,), blk.norm2.weight,
                                                blk.norm2.bias, 1e-6)
        assert relerr(blk.mlp(mlp_in), g["mlp"]) < TOL


def test_vit_golden(golden):
    g = golden("vit.pt")
    cfg = g["cfg"]
    m = asis.DinoVisionTransformer(img_size=cfg["img_size"], patch_size=14, embed_dim=cfg["embed_dim"], depth=cfg["depth"],
                                   num_heads=cfg["num_heads"], init_values=1e-5, block_chunks=0).to(DEV).eval()
    m.load_state_dict(g["sd"])
    img = g["img"].to(DEV)
    with asis.precision("fp32"), torch.no_grad():
        assert relerr(m.patch_embed(img), g["patch_tokens"]) < TOL
        taps = m.get_intermediate_layers(img, 4, return_class_token=True)
        for (a, b), (ga, gb) in zip(taps, g["taps"]):
            assert relerr(a, ga) < TOL and relerr(b, gb) < TOL
        nn_ = m.get_intermediate_layers(img, [1, 3], norm=False, reshape=True)
        for a, ga in zip(nn_, g["taps_nonorm"]):
            assert a.shape == ga.shape and relerr(a, ga) < TOL
        assert relerr(m(img), g["x_norm_clstoken"]) < TOL
        with pytest.raises(AssertionError, match="multiple of patch"):
            m.patch_embed(torch.rand(1, 3, 40, 42, device=DEV))


def test_adapter_blocks_golden(golden):
    g = golden("adapter.pt")
    dim, heads = g["cfg"]["dim"], g["cfg"]["heads"]
    x, c, gx, gc = [t.to(DEV) for t in adapter_data(dim)]
    inj = asis.CAViT(dim=dim, n_levels=3, num_heads=heads, n_points=4, init_values=0.0).to(DEV)
    ext = asis.CACNN(dim=dim, n_levels=1, num_heads=heads, n_points=4, cffn_ratio=0.25).to(DEV)
    d1, d2 = asis.deform_inputs(torch.zeros(1, 3, 588, 588, device=DEV), 14)
    with asis.precision("fp32"):
        # F4: the injector as constructed (gamma = 0) is a bit-exact identity
        with torch.no_grad():
            assert torch.equal(inj(x, d1[0], c, d1[1], d1[2]), x)
        inj.load_state_dict(g["inj_sd"])
        ext.load_state_dict(g["ext_sd"])
        xg = x.clone().requires_grad_(True)
        cg = c.clone().requires_grad_(True)
        x1 = inj(xg, d1[0], cg, d1[1], d1[2])
        c1 = ext(cg, d2[0], x1, d2[1], d2[2], 36, 36)
        assert relerr(x1, g["x1"]) < TOL and grad_err(c1, g["c1"]) < TOL
        ip, ep = dict(inj.named_parameters()), dict(ext.named_parameters())
        ni, ne = list(g["grad_inj"]), list(g["grad_ext"])
        grads = torch.autograd.grad([x1, c1], [xg, cg] + [ip[k] for k in ni] + [ep[k] for k in ne], [gx, gc])
        assert relerr(grads[0], g["grad_x"]) < TOL and grad_err(grads[1], g["grad_c"]) < TOL
        for k, gr in zip(ni, grads[2:2 + len(ni)]):
            assert relerr(gr, g["grad_inj"][k]) < GTOL, k
        for k, gr in zip(ne, grads[2 + len(ni):]):
            assert relerr(gr, g["grad_ext"][k]) < GTOL, k


def _build_encoder(g):
    cfg = g["cfg"]
    model = asis.DinoVisionTransformer(img_size=70, patch_size=14, embed_dim=cfg["dim"], depth=cfg["depth"],
                                       num_heads=cfg["heads"], init_values=1e-5, block_chunks=0).eval()
    enc = asis.AdapterEncoder(model=model, adapter_heads=cfg["heads"], inplanes=cfg["inplanes"]).to(DEV)
    enc.model.load_state_dict(g["vit_sd"])
    enc.backbone_encoder.load_state_dict(g["spm_sd"])
    enc.cross_vit.load_state_dict(g["inj_sd"])
    enc.cross_cnn.load_state_dict(g["ext_sd"])
    dec = asis.FeatureDecoder(embed_dim=cfg["dim"], num_classes=2, features=cfg["dec_features"]).to(DEV)
    dec.load_state_dict(g["dec_sd"])
    enc.backbone_encoder.train()
    dec.train()
    return enc, dec


def run_composed(g, mode):
    """Composed train.py data flow (encoder + decoder + loss) on the CUDA path in `mode`; returns internals and
    the gradients of loss + aux for every parameter the fixture lists."""
    cfg = g["cfg"]
    img, target, gfeat = [t.to(DEV) for t in encoder_data(1, 588, 3 * cfg["dim"], 42)]
    enc, dec = _build_encoder(g)
    with asis.precision(mode):
        res = enc(img)
        feat = res["feat"]
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=mode == "bf16"):     # as TrainStep.forward_loss does
            dl = dec(feat.float())
        logits = torch.nn.functional.interpolate(dl.float(), size=(588, 588), mode="bilinear")
        loss = o_enc.dice_loss(torch.softmax(logits, 1), target)
        aux = (feat * gfeat).sum() / feat.numel() ** 0.5
        named = {}
        for tag, mod in (("vit", enc.model), ("spm", enc.backbone_encoder), ("inj", enc.cross_vit),
                         ("ext", enc.cross_cnn), ("dec", dec)):
            for k, p in mod.named_parameters():
                named[f"{tag}.{k}"] = p
        keys = [k for k in g["grads"]]
        grads = torch.autograd.grad(loss + aux, [named[k] for k in keys], allow_unused=True)
    return dict(feat=feat, x=res["x"], logits=logits, loss=loss, grads=dict(zip(keys, grads)))


@pytest.mark.parametrize("fixture", ["encoder.pt", "encoder_hd64.pt"])
def test_composed_encoder_golden(golden, fixture):
    g = golden(fixture)
    r = run_composed(g, "fp32")
    assert grad_err(r["feat"], g["feat"]) < TOL
    assert grad_err(r["x"], g["x"]) < TOL
    logits = r["logits"]
    assert relerr(logits[:, :, ::12, ::12], g["logits_lowres"]) < TOL
    assert grad_err(logits[:, :, ::4, ::4], g["logits_s4"]) < TOL
    # the reference's argmax mask, EVERY pixel: bit-exact wherever the decision is numerically determined
    flips, near = mask_check(logits, g, TOL)
    print(f"[{fixture}] fp32 mode vs reference mask: {flips} flips / {logits[:, 0].numel()} pixels ({near} near-ties)")
    assert flips <= 3
    assert abs(float(r["loss"].detach()) - float(g["loss"])) < 1e-5
    checked = 0
    for k, gr in r["grads"].items():
        ref = g["grads"][k]
        assert gr is not None, k
        if not isinstance(ref, dict) and float(ref.abs().max()) < 1e-7:
            assert float(gr.abs().max()) < 1e-6, k
        else:
            # 1e-2: the reference's own fp32 gradients sit 1e-4..4.7e-3 from an fp64 evaluation of the same graph
            # (tests/test_oracle_golden.py::test_gradient_tolerance_is_fp32_summation_noise), so two correct fp32
            # evaluations can be twice that apart; the full-size test holds each gradient against fp64 instead
            assert grad_err(gr, ref) < 1e-2, k
        checked += 1
    assert checked > 100


def test_frozen_backbone_mode_matches_connected_forward(golden):
    """Reference wiring (backbone under no_grad, SURVEY.md F3): same forward values, no backbone grads."""
    g = golden("encoder.pt")
    cfg = g["cfg"]
    img, _, gfeat = [t.to(DEV) for t in encoder_data(1, 588, 3 * cfg["dim"], 42)]
    enc, _ = _build_encoder(g)
    enc.frozen_backbone = True
    with asis.precision("fp32"):
        res = enc(img)
        assert grad_err(res["feat"], g["feat"]) < TOL
        assert not res["feat"].requires_grad
