"""Seeded synthetic inputs and parameter initialisation shared by make_golden.py and the tests (no reference code
involved)."""
import torch

ENCODER_DATA_SEED = 1900


def synth_image(gen, B, size=588):
    """Deterministic 'frame': coarse random blocks + smooth ripple, values in [0,1)
    (the reference feeds un-normalised /255 pixels: tools/dataset.py:159)."""
    base = torch.rand(B, 3, size // 28, size // 28, generator=gen)
    img = base.repeat_interleave(28, 2).repeat_interleave(28, 3)
    t = torch.arange(size, dtype=torch.float32)
    ripple = 0.5 + 0.5 * torch.sin(t[:, None] * 0.071) * torch.cos(t[None, :] * 0.053)
    return (0.7 * img + 0.3 * ripple).clamp(0, 0.999)


def encoder_data(B=1, size=588, feat_channels=96, grid=42):
    gen = torch.Generator().manual_seed(ENCODER_DATA_SEED)
    img = synth_image(gen, B, size)
    target = (torch.rand(B, size, size, generator=gen) < 0.4).long()
    gfeat = torch.randn(B, feat_channels, grid, grid, generator=gen)
    return img, target, gfeat


def stress_init(module, gen, scaled=False):
    """Make every learnable path carry signal (default init leaves CAViT an identity, F4).
    ``scaled``: the two MSDA projections get std 1.5/sqrt(fan_in) and 1/sqrt(fan_in) (offsets ~1.5 px, attention
    logits ~1) instead of the fixed 0.3 / 0.5 of the dim-32 fixtures, which at larger widths would mean
    +-several px offsets and one-hot softmaxes -- a chaotic map rather than a trained adapter."""
    with torch.no_grad():
        for name, p in module.named_parameters():
            r = torch.randn(p.shape, generator=gen)
            fan = p.shape[-1] ** 0.5 if p.dim() > 1 else 1.0
            if name.endswith("gamma"):
                p.copy_(0.5 + 0.2 * r)
            elif "norm" in name and name.endswith("weight"):
                p.copy_(1.0 + 0.1 * r)
            elif "sampling_offsets.weight" in name:
                p.copy_((1.5 / fan if scaled else 0.3) * r)
            elif "attention_weights.weight" in name:
                p.copy_((1.0 / fan if scaled else 0.5) * r)
            elif name.endswith("bias") and "sampling_offsets" not in name:
                p.copy_(0.05 * r)
            elif name in ("cls_token", "mask_token"):
                p.copy_(0.1 * r)
    return module


ADAPTER_DATA_SEED = 1700


def adapter_data(dim, B=1, n_tok=1764, n_pyr=6949):
    gen = torch.Generator().manual_seed(ADAPTER_DATA_SEED)
    x = torch.randn(B, n_tok, dim, generator=gen)
    c = torch.randn(B, n_pyr, dim, generator=gen)
    gx = torch.randn(B, n_tok, dim, generator=gen)
    gc = torch.randn(B, n_pyr, dim, generator=gen)
    return x, c, gx, gc
