"""Generate the golden fixtures under tests/golden/ by running the REFERENCE's own modules.

Run in the build container only (the reference does not travel to the GPU box):

    PYTHONPATH=/root/reference XFORMERS_DISABLED=1 PYTHONDONTWRITEBYTECODE=1 \
        python tests/golden/make_golden.py

The reference ships no tests or golden vectors (SURVEY.md F8), so these fixtures -- outputs of
the unmodified reference classes on seeded inputs, CPU fp32 -- are what pins the oracle
(tests/test_oracle_golden.py) and, through it, the CUDA path.  Nothing from the reference's
source is written into the repo: only tensors.  Module weights, large outputs and the full-size logit margins
are packed by store.py (seed recipes checked by hash, digests, near-tie masks) so that every file stays under 1 MB.

Two deliberate deviations from "as shipped", both documented in SURVEY.md:
  * ``MSDeformAttnFunction`` has no backward (F2): for gradient fixtures its ``apply`` is
    re-pointed at the reference's own ``ms_deform_attn_core_pytorch`` (plain autograd);
  * ``nn.SyncBatchNorm`` cannot run on CPU: the spatial-prior module's SyncBN layers are
    converted to ``nn.BatchNorm2d`` with identical parameters (same state_dict keys, same
    training-mode batch statistics for world size 1).
"""
import os
import sys
import warnings

import torch
import torch.nn as nn

warnings.filterwarnings("ignore")
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, "/root/reference")
os.environ.setdefault("XFORMERS_DISABLED", "1")

from backbones.ops.modules import ms_deform_attn as ref_msda  # noqa: E402
from backbones import adapter_blocks as ref_ab  # noqa: E402
from backbones.encoders import FeatureEncoder  # noqa: E402
from backbones.decoders import FeatureDecoder  # noqa: E402
from dinov2.layers import MemEffAttention, NestedTensorBlock as Block  # noqa: E402
from dinov2.models import vision_transformer as ref_vits  # noqa: E402
from functools import partial  # noqa: E402

sys.path.insert(0, HERE)
from synth import adapter_data, encoder_data, stress_init  # noqa: E402
from store import digest, near_ties, pack_state_dicts  # noqa: E402


class _CoreApply:
    """Autograd-capable stand-in for MSDeformAttnFunction (see module docstring)."""

    @staticmethod
    def apply(value, shapes, lsi, loc, aw, im2col_step):
        return ref_msda.ms_deform_attn_core_pytorch(value, shapes, loc, aw)


def sync_bn_to_bn(module):
    for name, child in module.named_children():
        if isinstance(child, nn.SyncBatchNorm):
            bn = nn.BatchNorm2d(child.num_features, eps=child.eps, momentum=child.momentum)
            bn.load_state_dict(child.state_dict())
            setattr(module, name, bn)
        else:
            sync_bn_to_bn(child)
    return module


def cpu_sd(m):
    return {k: v.detach().clone() for k, v in m.state_dict().items()}


def save(name, obj):
    path = os.path.join(HERE, name)
    torch.save(obj, path)
    print(f"{name}: {os.path.getsize(path) / 1e3:.0f} kB")


def make_locs(gen, N, Lq, M, shapes, P, spread_px=3.0, oob_frac=0.08):
    """reference grid + U(-spread,spread) px, a fraction pushed outside [0,1] (zero-pad path)."""
    L = len(shapes)
    base = torch.rand(N, Lq, 1, 1, 1, 2, generator=gen)
    loc = base.expand(N, Lq, M, L, P, 2).clone()
    for l, (H, W) in enumerate(shapes):
        off = (torch.rand(N, Lq, M, P, 2, generator=gen) * 2 - 1) * spread_px
        loc[:, :, :, l] += off / torch.tensor([W, H], dtype=torch.float32)
    far = torch.rand(N, Lq, M, L, P, generator=gen) < oob_frac
    loc[far] = torch.rand(int(far.sum()), 2, generator=gen) * 1.6 - 0.3
    return loc


def gold_msda_core():
    cases = []
    specs = [
        dict(N=2, Lq=37, M=4, D=16, shapes=[(7, 9), (4, 5), (2, 3)], P=4),
        dict(N=1, Lq=50, M=3, D=12, shapes=[(6, 5)], P=2),           # non power-of-two head dim, single level
        dict(N=2, Lq=21, M=2, D=32, shapes=[(5, 5), (3, 4)], P=1),
    ]
    for i, sp in enumerate(specs):
        gen = torch.Generator().manual_seed(100 + i)
        shapes = sp["shapes"]
        S = sum(h * w for h, w in shapes)
        L = len(shapes)
        value = torch.randn(sp["N"], S, sp["M"], sp["D"], generator=gen, requires_grad=True)
        loc = make_locs(gen, sp["N"], sp["Lq"], sp["M"], shapes, sp["P"]).requires_grad_(True)
        aw = torch.softmax(torch.randn(sp["N"], sp["Lq"], sp["M"], L * sp["P"], generator=gen), -1)
        aw = aw.view(sp["N"], sp["Lq"], sp["M"], L, sp["P"]).clone().requires_grad_(True)
        ss = torch.as_tensor(shapes, dtype=torch.long)
        out = ref_msda.ms_deform_attn_core_pytorch(value, ss, loc, aw)
        gout = torch.randn(out.shape, generator=gen)
        gv, gl, ga = torch.autograd.grad(out, (value, loc, aw), gout)
        # forward through the as-shipped Function too (it has a forward)
        lsi = torch.cat([ss.new_zeros(1), ss.prod(1).cumsum(0)[:-1]])
        out_fn = ref_msda.MSDeformAttnFunction.apply(value.detach(), ss, lsi, loc.detach(), aw.detach(), 64)
        assert torch.equal(out_fn, out.detach())
        cases.append(dict(spatial_shapes=ss, level_start_index=lsi, value=value.detach(), loc=loc.detach(),
                          aw=aw.detach(), out=out.detach(), grad_out=gout, grad_value=gv, grad_loc=gl, grad_aw=ga))
    save("msda_core.pt", cases)


def gold_msda_module():
    gen = torch.Generator().manual_seed(7)
    torch.manual_seed(7)
    m = ref_msda.MSDeformAttn(d_model=32, n_levels=3, n_heads=4, n_points=4, ratio=1.0)
    default_bias = m.sampling_offsets.bias.detach().clone()
    stress_init(m, gen)
    shapes = [(9, 9), (4, 4), (2, 2)]
    ss = torch.as_tensor(shapes, dtype=torch.long)
    lsi = torch.cat([ss.new_zeros(1), ss.prod(1).cumsum(0)[:-1]])
    S = int(ss.prod(1).sum())
    N, Lq = 2, 25
    query = torch.randn(N, Lq, 32, generator=gen)
    feat = torch.randn(N, S, 32, generator=gen)
    ref = ref_ab.get_reference_points([(5, 5)], "cpu")                    # [1,25,1,2]
    out = m(query, ref, feat, ss, lsi, None)
    mask = torch.rand(N, S, generator=gen) < 0.2
    out_masked = m(query, ref, feat, ss, lsi, mask)
    ref4 = torch.cat([ref.expand(N, Lq, 3, 2), torch.rand(N, Lq, 3, 2, generator=gen) * 0.3], -1)
    out_box = m(query, ref4, feat, ss, lsi, None)
    save("msda_module.pt", dict(cfg=dict(d_model=32, n_levels=3, n_heads=4, n_points=4, ratio=1.0), sd=cpu_sd(m),
                                default_bias=default_bias, spatial_shapes=ss, level_start_index=lsi, query=query,
                                feat=feat, ref=ref, out=out.detach(), mask=mask, out_masked=out_masked.detach(),
                                ref4=ref4, out_box=out_box.detach()))


def gold_block():
    gen = torch.Generator().manual_seed(11)
    torch.manual_seed(11)
    blk = Block(dim=64, num_heads=4, mlp_ratio=4.0, qkv_bias=True, proj_bias=True, ffn_bias=True,
                init_values=1e-5, norm_layer=partial(nn.LayerNorm, eps=1e-6), attn_class=MemEffAttention)
    blk.eval()
    stress_init(blk, gen)
    x = torch.randn(2, 19, 64, generator=gen, requires_grad=True)
    y = blk(x)
    gy = torch.randn(y.shape, generator=gen)
    params = dict(blk.named_parameters())
    grads = torch.autograd.grad(y, [x] + list(params.values()), gy)
    # pieces, for op-level tests
    ln1 = blk.norm1(x)
    att = blk.attn(ln1)
    ln2_in = x + blk.ls1(att)
    mlp_out = blk.mlp(blk.norm2(ln2_in))
    save("block.pt", dict(cfg=dict(dim=64, num_heads=4), sd=cpu_sd(blk), x=x.detach(), y=y.detach(), grad_y=gy,
                          grad_x=grads[0], grad_params={k: g for k, g in zip(params.keys(), grads[1:])},
                          ln1=ln1.detach(), attn=att.detach(), mlp=mlp_out.detach()))


def tiny_vit(embed_dim, depth, heads, gen, img_size=28):
    m = ref_vits.DinoVisionTransformer(img_size=img_size, patch_size=14, embed_dim=embed_dim, depth=depth,
                                       num_heads=heads, mlp_ratio=4, init_values=1e-5, ffn_layer="mlp",
                                       block_chunks=0, block_fn=partial(Block, attn_class=MemEffAttention))
    m.eval()
    return stress_init(m, gen)


def gold_vit():
    gen = torch.Generator().manual_seed(13)
    torch.manual_seed(13)
    m = tiny_vit(64, 5, 4, gen)
    img = torch.rand(2, 3, 42, 42, generator=gen)
    with torch.no_grad():
        taps = m.get_intermediate_layers(img, 4, return_class_token=True)
        taps_nonorm = m.get_intermediate_layers(img, [1, 3], norm=False, reshape=True)
        pe = m.interpolate_pos_encoding(torch.zeros(1, 10, 64), 42, 42)
        tok = m.patch_embed(img)
        feats = m.forward_features(img)
    fx = dict(cfg=dict(embed_dim=64, depth=5, num_heads=4, patch=14, img_size=28), sd=cpu_sd(m), img=img,
              taps=[(a.clone(), b.clone()) for a, b in taps], taps_nonorm=[t.clone() for t in taps_nonorm],
              pos=pe.clone(), patch_tokens=tok.clone(), x_norm_clstoken=feats["x_norm_clstoken"].clone())
    pack_state_dicts(fx, dict(kind="vit", seed=13, dim=64, depth=5, heads=4, img_size=28), ["sd"])
    save("vit.pt", fx)


def gold_adapter():
    gen = torch.Generator().manual_seed(17)
    torch.manual_seed(17)
    dim, heads = 32, 4
    inj = ref_ab.CAViT(dim=dim, n_levels=3, num_heads=heads, n_points=4, init_values=0.0)
    ext = ref_ab.CACNN(dim=dim, n_levels=1, num_heads=heads, n_points=4, with_cffn=True, cffn_ratio=0.25)
    d1, d2 = ref_ab.deform_inputs(torch.zeros(1, 3, 588, 588), 14)
    x, c, gx, gc = adapter_data(dim)
    with torch.no_grad():
        ident = inj(x, d1[0], c, d1[1], d1[2])
    assert torch.equal(ident, x)                         # F4: default injector is an identity
    stress_init(inj, gen)
    stress_init(ext, gen)
    old = ref_msda.MSDeformAttnFunction
    ref_msda.MSDeformAttnFunction = _CoreApply
    try:
        xg = x.clone().requires_grad_(True)
        cg = c.clone().requires_grad_(True)
        x1 = inj(xg, d1[0], cg, d1[1], d1[2])
        c1 = ext(cg, d2[0], x1, d2[1], d2[2], 36, 36)
        inj_p = dict(inj.named_parameters())
        ext_p = dict(ext.named_parameters())
        grads = torch.autograd.grad([x1, c1], [xg, cg] + list(inj_p.values()) + list(ext_p.values()), [gx, gc])
    finally:
        ref_msda.MSDeformAttnFunction = old
    n1 = len(inj_p)
    save("adapter.pt", dict(cfg=dict(dim=dim, heads=heads), inj_sd=cpu_sd(inj), ext_sd=cpu_sd(ext),
                            d1=[t.clone() for t in d1], d2=[t.clone() for t in d2], x_sum=x.double().sum(), c_sum=c.double().sum(),
                            x1=x1.detach(), c1=digest(c1),
                            grad_x=grads[0], grad_c=digest(grads[1]),
                            grad_inj={k: g for k, g in zip(inj_p.keys(), grads[2:2 + n1])},
                            grad_ext={k: g for k, g in zip(ext_p.keys(), grads[2 + n1:])}))


def gold_encoder(name="encoder.pt", dim=32, heads=2, depth=5, seed=19, full_grad_numel=4096, scaled=False, amp=False):
    """train.py:275-406 data flow with the reference's own modules, graph left connected.
    ``encoder.pt``: head_dim 16 (fp32 parity mode).  ``encoder_hd64.pt``: head_dim 64 for the backbone AND
    the adapters (dim 128, 2 heads), the shape class the tcgen05 attention / bf16 MSDA kernels need, so the
    bf16 performance mode can be compared with the reference end to end.
    Near-tie masks are stored at 1e-4 (fp32 parity) and, with ``amp``, at the bf16 mode's logit tolerance
    max(2e-2, the reference's own bf16-autocast logit error)."""
    from einops import rearrange
    import torch.nn.functional as F
    import numpy as np
    gen = torch.Generator().manual_seed(seed)
    torch.manual_seed(seed)
    model = tiny_vit(dim, depth, heads, gen, img_size=70)
    enc = stress_init(sync_bn_to_bn(FeatureEncoder(inplanes=8, embed_dim=dim)), gen)
    inj = stress_init(ref_ab.CAViT(dim=dim, n_levels=3, num_heads=heads, n_points=4, init_values=0.0), gen, scaled)
    ext = stress_init(ref_ab.CACNN(dim=dim, n_levels=1, num_heads=heads, n_points=4, cffn_ratio=0.25), gen, scaled)
    dec = stress_init(FeatureDecoder(embed_dim=dim, num_classes=2, features=[dim, 16, 8, 8, 4]), gen)
    enc.train(); dec.train()
    inp, target, gfeat = encoder_data(1, 588, 3 * dim, 42)
    old = ref_msda.MSDeformAttnFunction
    ref_msda.MSDeformAttnFunction = _CoreApply

    def run():
        d1, d2 = ref_ab.deform_inputs(inp, 14)
        c1, c2, c3, c4 = enc(inp)
        c = torch.cat([c2, c3, c4], dim=1)
        with torch.no_grad():
            taps = model.get_intermediate_layers(inp, 4, return_class_token=True)
            taps = [t for t, _ in taps]
        x = model.patch_embed(inp)
        for blk in model.blocks[0:-3]:
            x = blk(x)
        for stage in range(4):
            if stage > 0:
                x = model.blocks[depth - 4 + stage](x)
            x = inj(query=x, reference_points=d1[0], feat=c, spatial_shapes=d1[1], level_start_index=d1[2])
            c = ext(query=c, reference_points=d2[0], feat=x, spatial_shapes=d2[1], level_start_index=d2[2], H=36, W=36)
            x = x + taps[stage]
        out_last = rearrange(x, "b (h w) c -> b c h w", h=42, w=42)
        out_vit = rearrange(taps[3], "b (h w) c -> b c h w", h=42, w=42)
        c4m = rearrange(c4, "b (h w) c -> b c h w", h=18, w=18)
        c4m = F.pad(c4m, [12, 12, 12, 12])
        feat = torch.cat((out_last, c4m, out_vit), dim=1)
        logits = dec(feat)
        logits = F.interpolate(logits, size=(588, 588), mode="bilinear")
        prob = nn.Softmax(1)(logits)
        # DC(2).forward restated inline because the reference's onehot() calls .cuda()
        p2 = torch.softmax(prob, 1)
        onehot = torch.zeros_like(p2).scatter_(1, target.unsqueeze(1), 1.0)
        inter = (p2 * onehot).sum((2, 3))
        loss = 1.0 - ((2 * inter) / (p2.sum((2, 3)) + onehot.sum((2, 3)) + 10e-20)).mean()
        named = {}
        for tag, mod in (("vit", model), ("spm", enc), ("inj", inj), ("ext", ext), ("dec", dec)):
            for k, p in mod.named_parameters():
                named[f"{tag}.{k}"] = p
        # a second scalar that exercises the encoder graph directly (the dice loss of a
        # 2-class softmax-of-softmax is very flat)
        aux = (feat * gfeat).sum() / feat.numel() ** 0.5
        grads = torch.autograd.grad(loss + aux, list(named.values()), allow_unused=True)
        return x, c, feat, logits, loss, aux, named, grads

    amp_err = None
    try:
        x, c, feat, logits, loss, aux, named, grads = run()
        if amp:
            # How far the REFERENCE ITSELF moves when PyTorch runs it in bf16 mixed precision (torch.autocast, what
            # train.py does with fp16 around feature_model): the yardstick for "bf16 mode" gradient tolerances.
            with torch.autocast("cpu", dtype=torch.bfloat16):
                xa, ca, feata, logitsa, lossa, auxa, _, gradsa = run()

            def rel(a, b):
                return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))
            amp_err = dict(x=rel(xa, x), feat=rel(feata, feat), logits=rel(logitsa, logits),
                           loss=abs(float(lossa) - float(loss)),
                           grads={k: rel(ga, g) for k, g, ga in zip(named, grads, gradsa)
                                  if g is not None and float(g.abs().max()) > 1e-7})
    finally:
        ref_msda.MSDeformAttnFunction = old
    gsel = {}
    for (k, p), g in zip(named.items(), grads):
        if g is None:
            continue
        gsel[k] = g if g.numel() <= full_grad_numel else digest(g)
    mask = logits.argmax(1).to(torch.uint8).numpy()                      # [1, 588, 588] in {0, 1}
    logits_absmax = float(logits.detach().abs().max())
    # class-1 minus class-0 logit at every pixel (fp16 is plenty: it only tells the tests which pixels are numerical
    # near-ties, where two correct evaluations may legitimately disagree)
    margin = (logits.detach()[:, 1] - logits.detach()[:, 0]).half()
    tols = (1e-4,) + ((max(2e-2, amp_err["logits"]),) if amp else ())
    fx = dict(cfg=dict(dim=dim, heads=heads, depth=depth, inplanes=8, dec_features=[dim, 16, 8, 8, 4]),
              vit_sd=cpu_sd(model), spm_sd=cpu_sd(enc), inj_sd=cpu_sd(inj), ext_sd=cpu_sd(ext),
              dec_sd=cpu_sd(dec), img_lowres=inp[:, :, ::28, ::28].clone(),
              img_sum=inp.double().sum(), target_sum=int(target.sum()),
              feat=digest(feat), x=digest(x), c_sum=c.detach().double().sum(),
              logits_lowres=logits.detach()[:, :, ::12, ::12].clone(),
              logits_s4=digest(logits[:, :, ::4, ::4]),
              argmax_sum=int(logits.argmax(1).sum()),
              argmax_packed=torch.from_numpy(np.packbits(mask.reshape(-1))), argmax_shape=tuple(mask.shape),
              near_ties=near_ties(margin, logits_absmax, tols), logits_absmax=logits_absmax,
              loss=loss.detach(), aux=aux.detach(), grads=gsel, amp_err=amp_err)
    pack_state_dicts(fx, dict(kind="encoder", seed=seed, dim=dim, heads=heads, depth=depth, inplanes=8,
                              dec_features=[dim, 16, 8, 8, 4], scaled=scaled),
                     ["vit_sd", "spm_sd", "inj_sd", "ext_sd", "dec_sd"])
    save(name, fx)


def _reference_mask_transformer():
    """The reference's ``MaskTransformer`` class object, built from its unmodified source text.
    backbones/masktrans_block.py imports ``timm`` (absent here) for DropPath only -- which the reference instantiates
    with drop_path 0.0, i.e. never: a stand-in module named ``timm.models.layers`` supplies the name; the evaluation
    script itself imports torchmetrics / dataset tooling at module level, so only its ``init_weights`` function and
    ``MaskTransformer`` class nodes (eval/eval_dinov2_masktrans.py:389-480) are compiled, from the file's own text."""
    import ast
    import types
    for name in ("timm", "timm.models", "timm.models.layers"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["timm.models.layers"].DropPath = ref_ab.DropPath          # the reference's own local DropPath (adapter_blocks.py:41-60)
    sys.modules["timm.models.layers"].trunc_normal_ = nn.init.trunc_normal_
    from backbones.masktrans_block import Block as MTBlock
    path = "/root/reference/eval/eval_dinov2_masktrans.py"
    tree = ast.parse(open(path).read())
    keep = [n for n in tree.body if isinstance(n, (ast.FunctionDef, ast.ClassDef)) and n.name in ("init_weights", "MaskTransformer")]
    assert len(keep) == 2
    from einops import rearrange
    ns = dict(torch=torch, nn=nn, Block=MTBlock, trunc_normal_=nn.init.trunc_normal_, rearrange=rearrange)
    exec(compile(ast.Module(body=keep, type_ignores=[]), path, "exec"), ns)
    return ns["MaskTransformer"]


def gold_masktrans():
    """BASELINE config[3]'s decoder: MaskTransformer(n_cls=8) on a [B, 36, d] token grid (6 x 6 patches of 14 px),
    eval mode (dropout = identity), logits resized to the image and arg-maxed as validate_network does (:361-366)."""
    MaskTransformer = _reference_mask_transformer()
    gen = torch.Generator().manual_seed(29)
    torch.manual_seed(29)
    d, heads, n_cls, gs, B = 128, 2, 8, 6, 2
    m = MaskTransformer(n_cls=n_cls, patch_size=14, d_encoder=d, n_layers=2, n_heads=heads, d_model=d, d_ff=4 * d,
                        drop_path_rate=0.0, dropout=0.1)
    stress_init(m, gen)
    with torch.no_grad():
        m.cls_emb.copy_(0.5 * torch.randn(m.cls_emb.shape, generator=gen))
    m.eval()
    x = torch.randn(B, gs * gs, d, generator=gen)
    im = (gs * 14, gs * 14)
    with torch.no_grad():
        masks = m(x, im)
        out = torch.nn.functional.interpolate(masks, size=im, mode="bilinear")
        pred = torch.softmax(out, dim=1).argmax(1)
    # gradients too (the reference trains this decoder, eval_dinov2_masktrans.py:262-300), dropout still off
    xg = x.clone().requires_grad_(True)
    gy = torch.randn(masks.shape, generator=gen)
    mg = m(xg, im)
    grads = torch.autograd.grad(mg, [xg] + list(m.parameters()), gy)
    names = ["input"] + [n for n, _ in m.named_parameters()]
    fx = dict(cfg=dict(d=d, heads=heads, n_cls=n_cls, gs=gs), sd=cpu_sd(m), x=x, masks=masks, logits=out,
              pred=pred.to(torch.uint8), gy=gy, grads={n: g if g.numel() <= 4096 else digest(g) for n, g in zip(names, grads)})
    pack_state_dicts(fx, dict(kind="masktrans", seed=29, d=d, heads=heads, n_cls=n_cls), ["sd"])
    save("masktrans.pt", fx)


if __name__ == "__main__":
    gold_masktrans()
    gold_msda_core()
    gold_msda_module()
    gold_block()
    gold_vit()
    gold_adapter()
    gold_encoder()
    gold_encoder("encoder_hd64.pt", dim=128, heads=2, depth=5, seed=23, scaled=True, amp=True)
