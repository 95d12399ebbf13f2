"""Attention kernel microbench at the step's shape (B=12, T=1765, H=16, hd=64): forward and backward, CUDA events,
median of N, checked against fp32 math on one (image, head) slice."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from adaptersis_b200 import kernels as K  # noqa: E402
from adaptersis_b200._lib import BF16  # noqa: E402

B, T, H = (int(x) for x in (sys.argv[1:4] if len(sys.argv) > 3 else (12, 1765, 16)))
dev = torch.device("cuda:0")
g = torch.Generator().manual_seed(0)
qkv = (torch.randn(B, T, 3 * H * 64, generator=g) * 0.7).to(dev).bfloat16()
out, lse = K.attention_forward(BF16, qkv, B, T, H, 64)
dout = torch.randn(out.shape, generator=g).to(dev).bfloat16()


def med(fn, n=15):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2]


tf = med(lambda: K.attention_forward(BF16, qkv, B, T, H, 64))
tb = med(lambda: K.attention_backward(BF16, qkv, out, lse, dout, B, T, H, 64))
# correctness on the last image / head (includes the ragged last tiles)
b, h = B - 1, H - 1
x = qkv[b].float().view(T, 3, H, 64)
q, k, v = x[:, 0, h], x[:, 1, h], x[:, 2, h]
s = (q * 64 ** -0.5) @ k.t()
ref = torch.softmax(s, -1) @ v
err = float((out[b, :, h * 64:(h + 1) * 64].float() - ref).abs().max() / ref.abs().max())
lerr = float((lse[b, h] - torch.logsumexp(s, -1)).abs().max())
out2, lse2 = K.attention_forward(BF16, qkv, B, T, H, 64)
fl = 4.0 * B * H * T * T * 64
print(json.dumps(dict(B=B, T=T, H=H, fwd_us=round(tf * 1e3, 1), fwd_tflops=round(fl / tf / 1e9, 1), bwd_us=round(tb * 1e3, 1),
                      bwd_tflops_alg=round(2.5 * fl / tb / 1e9, 1), out_relerr=round(err, 5), lse_abserr=round(lerr, 6),
                      finite=bool(torch.isfinite(out.float()).all()), repeatable=bool(torch.equal(out, out2) and torch.equal(lse, lse2)))))
