"""How the golden fixtures are stored: make_golden.py packs them, conftest.load_golden unpacks them.

Each fixture file stays under 1 MB, so three kinds of entry are not stored verbatim:
  * state dicts of the stress-initialised modules: the fixture keeps the seed recipe, an SHA-256 of every tensor the
    reference produced and the BatchNorm running statistics; `unpack` rebuilds the modules with adaptersis_b200's
    constructors (which draw from the random stream in the reference's order) and refuses a rebuilt tensor whose
    hash differs, so a loaded fixture is bit-identical to what the reference made;
  * large outputs and gradients: a digest {norm, sum, absmax, head, sample} (conftest.grad_err compares with it);
  * the class-1 minus class-0 margin of a full-size mask: only the near-tie pixels at each tolerance a test uses,
    bit-packed (conftest.mask_check).
"""
import hashlib
from functools import partial

import numpy as np
import torch

from synth import stress_init


def sample_idx(numel, n=4096):
    """Evenly strided sample positions of a flattened tensor."""
    step = max(1, numel // n)
    return torch.arange(0, numel, step)[:n]


def digest(t, n=4096):
    t = t.detach()
    return dict(norm=float(t.double().norm()), head=t.flatten()[:256].clone(), sum=float(t.double().sum()),
                sample=t.flatten()[sample_idx(t.numel(), n)].clone(), absmax=float(t.abs().max()))


def tensor_sha256(t):
    t = t.detach().contiguous().cpu()
    h = hashlib.sha256(f"{t.dtype}{tuple(t.shape)}".encode())
    h.update(t.numpy().tobytes())
    return h.hexdigest()


def _is_stat(key):
    return "running_" in key or key.endswith("num_batches_tracked")


def pack_state_dicts(fixture, recipe, keys):
    """Replace the state dicts fixture[k] (k in keys) by `recipe` + hashes + BatchNorm statistics."""
    sha, stats = {}, {}
    for k in keys:
        sd = fixture.pop(k)
        sha[k] = {n: tensor_sha256(v) for n, v in sd.items()}
        stats[k] = {n: v.clone() for n, v in sd.items() if _is_stat(n)}
    fixture["weights"] = dict(recipe=recipe, sha256=sha, stats=stats)


def near_ties(margin, logits_absmax, tols):
    """{tol: bit-packed mask of the pixels whose margin is a numerical near-tie at `tol`} (see conftest.mask_check)."""
    m = margin.float().abs()
    return {float(t): torch.from_numpy(np.packbits((m <= 2 * t * logits_absmax + 1e-3 * m).numpy().reshape(-1)))
            for t in tols}


def _tiny_vit(asis, dim, depth, heads, gen, img_size):
    m = asis.DinoVisionTransformer(img_size=img_size, patch_size=14, embed_dim=dim, depth=depth, num_heads=heads,
                                   mlp_ratio=4, init_values=1e-5, ffn_layer="mlp", block_chunks=0,
                                   block_fn=partial(asis.Block, attn_class=asis.MemEffAttention))
    m.eval()
    return stress_init(m, gen)


def build_modules(recipe):
    """The modules make_golden.py built for `recipe`, from adaptersis_b200's constructors: {fixture key: module}."""
    import adaptersis_b200 as asis
    r = dict(recipe)
    kind, seed = r.pop("kind"), r.pop("seed")
    gen = torch.Generator().manual_seed(seed)
    torch.manual_seed(seed)
    if kind == "vit":
        return {"sd": _tiny_vit(asis, r["dim"], r["depth"], r["heads"], gen, r["img_size"])}
    if kind == "encoder":
        dim, heads, scaled = r["dim"], r["heads"], r["scaled"]
        mods = {"vit_sd": _tiny_vit(asis, dim, r["depth"], heads, gen, 70)}
        mods["spm_sd"] = stress_init(asis.FeatureEncoder(inplanes=r["inplanes"], embed_dim=dim), gen)
        mods["inj_sd"] = stress_init(asis.CAViT(dim=dim, n_levels=3, num_heads=heads, n_points=4, init_values=0.0), gen,
                                     scaled)
        mods["ext_sd"] = stress_init(asis.CACNN(dim=dim, n_levels=1, num_heads=heads, n_points=4, cffn_ratio=0.25), gen,
                                     scaled)
        mods["dec_sd"] = stress_init(asis.FeatureDecoder(embed_dim=dim, num_classes=2, features=r["dec_features"]), gen)
        return mods
    if kind == "masktrans":
        d = r["d"]
        m = asis.MaskTransformer(n_cls=r["n_cls"], patch_size=14, d_encoder=d, n_layers=2, n_heads=r["heads"], d_model=d,
                                 d_ff=4 * d, drop_path_rate=0.0, dropout=0.1)
        stress_init(m, gen)
        with torch.no_grad():
            m.cls_emb.copy_(0.5 * torch.randn(m.cls_emb.shape, generator=gen))
        return {"sd": m}
    raise ValueError(f"unknown fixture recipe {kind!r}")


def unpack(fixture):
    """Rebuild the state dicts of a packed fixture in place; every tensor must hash to the reference's."""
    if not isinstance(fixture, dict) or "weights" not in fixture:
        return fixture
    w = fixture.pop("weights")
    with torch.random.fork_rng(devices=[]):
        mods = build_modules(w["recipe"])
    for key, m in mods.items():
        sd = {n: v.detach().clone() for n, v in m.state_dict().items()}
        sd.update(w["stats"][key])
        want = w["sha256"][key]
        bad = sorted(set(sd) ^ set(want)) + [n for n in want if n in sd and tensor_sha256(sd[n]) != want[n]]
        if bad:
            raise RuntimeError(f"golden {key}: rebuilt tensors differ from the reference's: {bad[:8]}")
        fixture[key] = sd
    return fixture
