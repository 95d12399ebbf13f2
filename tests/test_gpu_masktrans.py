"""BASELINE config[3]: the mask-transformer decoder (eval/eval_dinov2_masktrans.py:400-465) on the CUDA path, against the
fixture produced by the reference's own class (tests/golden/make_golden.py::gold_masktrans) -- logits, the resized logits,
the arg-max prediction and every gradient -- in both precision modes.  Tolerances: fp32 mode 1e-4 (parameter gradients
1e-3), prediction bit-exact; bf16 mode 2e-2 (gradients 3e-2), prediction identical wherever the top-2 logit margin exceeds
the tolerance granted to the logits."""
import pytest
import torch
import torch.nn.functional as F

from conftest import grad_err, relerr

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _build(g):
    from adaptersis_b200.masktrans import MaskTransformer
    c = g["cfg"]
    m = MaskTransformer(n_cls=c["n_cls"], patch_size=14, d_encoder=c["d"], n_layers=2, n_heads=c["heads"], d_model=c["d"],
                        d_ff=4 * c["d"], drop_path_rate=0.0, dropout=0.1).to(DEV)
    m.load_state_dict(g["sd"], strict=True)
    return m.eval(), (c["gs"] * 14, c["gs"] * 14)


@pytest.mark.parametrize("mode,tol,gtol", [("fp32", 1e-4, 1e-3), ("bf16", 2e-2, 3e-2)])
def test_mask_transformer_golden(golden, mode, tol, gtol):
    import adaptersis_b200 as asis
    g = golden("masktrans.pt")
    m, im = _build(g)
    x = g["x"].to(DEV).requires_grad_(True)
    names = [n for n in g["grads"] if n != "input"]
    with asis.precision(mode):
        masks = m(x, im)
        grads = torch.autograd.grad(masks, [x] + [dict(m.named_parameters())[n] for n in names], g["gy"].to(DEV))
    assert masks.shape == g["masks"].shape and relerr(masks.float(), g["masks"]) < tol
    out = F.interpolate(masks.float(), size=im, mode="bilinear")
    assert relerr(out, g["logits"]) < tol
    pred = torch.softmax(out, 1).argmax(1).to(torch.uint8).cpu()
    top2 = g["logits"].topk(2, dim=1).values
    margin = top2[:, 0] - top2[:, 1]
    decided = margin > 2 * tol * float(g["logits"].abs().max())
    if mode == "fp32":
        assert torch.equal(pred, g["pred"])                                 # bit-exact
    assert torch.equal(pred[decided], g["pred"][decided])
    bad = [(n, grad_err(a, g["grads"][n])) for n, a in zip(["input"] + names, grads) if not grad_err(a, g["grads"][n]) < gtol]
    assert not bad, bad


def test_training_mode_dropout_is_rejected(golden):
    g = golden("masktrans.pt")
    m, im = _build(g)
    m.train()
    with pytest.raises(NotImplementedError):
        m(g["x"].to(DEV), im)
