import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def load_golden(name):
    from store import unpack
    return unpack(torch.load(os.path.join(GOLDEN, name), map_location="cpu", weights_only=False))


@pytest.fixture(scope="session")
def golden():
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = load_golden(name)
        return cache[name]

    return get


def relerr(a, b):
    """max |a-b| / max |b|  -- the 'max relative error' used throughout (tolerance stated per test)."""
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def relerr_rms(a, b):
    """max |a-b| / rms(b): the same error held against the TYPICAL magnitude instead of the largest one
    (4-6x stricter than relerr for activation-like tensors); reported next to relerr in the parity tables."""
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    return float((a - b).abs().max() / b.pow(2).mean().sqrt().clamp_min(1e-30))


def unpack_mask(g):
    """The reference's full argmax mask stored bit-packed in a composed-encoder fixture -> uint8 [B,H,W]."""
    import numpy as np
    shape = tuple(g["argmax_shape"])
    n = 1
    for d in shape:
        n *= d
    bits = np.unpackbits(g["argmax_packed"].numpy())[:n]
    return torch.from_numpy(bits.reshape(shape))


def sample_idx(numel, n=4096):
    step = max(1, numel // n)
    return torch.arange(0, numel, step)[:n]


def grad_err(gr, ref):
    """Error of a tensor against its fixture entry (full tensor, or {norm, head, sample, absmax} for big ones),
    normalised by the reference tensor's largest magnitude."""
    gr = gr.detach().float().cpu()
    if not isinstance(ref, dict):
        return relerr(gr, ref)
    scale = float(ref["absmax"]) if "absmax" in ref else float(ref["head"].abs().max())
    scale = max(scale, 1e-30)
    e = float((gr.flatten()[:256] - ref["head"]).abs().max()) / scale
    if "sample" in ref:
        idx = sample_idx(gr.numel(), ref["sample"].numel())
        e = max(e, float((gr.flatten()[idx] - ref["sample"]).abs().max()) / scale)
    e = max(e, abs(float(gr.double().norm()) - float(ref["norm"])) / (float(ref["norm"]) + 1e-30))
    return e


def mask_check(logits, g, tol):
    """Argmax segmentation mask against the reference's, pixel by pixel.  Returns (flips, near_ties).
    Every pixel whose reference decision is numerically determined -- |logit1 - logit0| above 2 x `tol` x max|logit|:
    `tol` is what north_star grants EACH logit, and the margin is a difference of two -- must agree BIT-EXACTLY; at the remaining near-tie
    pixels two correct evaluations (even the reference run with another summation order) can differ, so flips
    there are counted and reported, not hidden.  The fixture stores the near-tie pixels at each `tol` a test uses
    (tests/golden/store.py)."""
    import numpy as np
    ours = logits.detach().argmax(1).to(torch.uint8).cpu()
    ref = unpack_mask(g)
    flips = ours != ref
    if tol not in g["near_ties"]:
        raise KeyError(f"the fixture stores near-tie masks at tolerances {sorted(g['near_ties'])}, not at {tol}")
    near = torch.from_numpy(np.unpackbits(g["near_ties"][tol].numpy())[:ref.numel()].reshape(ref.shape)).bool()
    bad = flips & ~near
    assert not bool(bad.any()), f"{int(bad.sum())} argmax flips at numerically determined pixels"
    return int(flips.sum()), int(near.sum())


def as_fixture_entry(truth, like):
    """Put a full 'truth' gradient into the shape of the fixture entry `like` (full tensor, or the
    {norm, head, sample, absmax} digest stored for big tensors) so that grad_err measures both the same way."""
    t = truth.detach().float().cpu()
    if not isinstance(like, dict):
        return t
    return dict(norm=t.double().norm(), head=t.flatten()[:256].clone(), sample=t.flatten()[sample_idx(t.numel())].clone(),
                absmax=t.abs().max())
