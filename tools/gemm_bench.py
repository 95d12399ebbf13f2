"""Per-shape microbench of the tcgen05 GEMM on the shapes of the ViT-L/14 training step (the rows of
`bench.py --detail`): TFLOP/s per launch, CUDA events on the launching stream, inputs larger than L2."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from adaptersis_b200 import kernels as K  # noqa: E402
from adaptersis_b200._lib import (BF16, EPI_DGELU, EPI_GELU, EPI_NONE, EPI_SCALE_RESIDUAL, MAJOR_K, MAJOR_MN)  # noqa: E402

R = 21180
# name, M, N, K, a_major, b_major, epilogue, out dtype, aux, bias
SHAPES = [
    ("qkv fwd", R, 3072, 1024, MAJOR_K, MAJOR_K, EPI_NONE, torch.bfloat16, False, True),
    ("proj fwd +res", R, 1024, 1024, MAJOR_K, MAJOR_K, EPI_SCALE_RESIDUAL, torch.float32, True, True),
    ("fc1 fwd +gelu", R, 4096, 1024, MAJOR_K, MAJOR_K, EPI_GELU, torch.bfloat16, True, True),
    ("fc1 fwd +gelu (taps, no aux)", R, 4096, 1024, MAJOR_K, MAJOR_K, EPI_GELU, torch.bfloat16, False, True),
    ("fc2 fwd +res", R, 1024, 4096, MAJOR_K, MAJOR_K, EPI_SCALE_RESIDUAL, torch.float32, True, True),
    ("fc2 dgrad +dgelu", R, 4096, 1024, MAJOR_K, MAJOR_MN, EPI_DGELU, torch.bfloat16, True, False),
    ("fc1 dgrad", R, 1024, 4096, MAJOR_K, MAJOR_MN, EPI_NONE, torch.bfloat16, False, False),
    ("qkv dgrad", R, 1024, 3072, MAJOR_K, MAJOR_MN, EPI_NONE, torch.bfloat16, False, False),
    ("proj dgrad", R, 1024, 1024, MAJOR_K, MAJOR_MN, EPI_NONE, torch.bfloat16, False, False),
    ("fc1 wgrad", 4096, 1024, R, MAJOR_MN, MAJOR_MN, EPI_NONE, torch.float32, False, False),
    ("fc2 wgrad", 1024, 4096, R, MAJOR_MN, MAJOR_MN, EPI_NONE, torch.float32, False, False),
    ("qkv wgrad", 3072, 1024, R, MAJOR_MN, MAJOR_MN, EPI_NONE, torch.float32, False, False),
    ("proj wgrad", 1024, 1024, R, MAJOR_MN, MAJOR_MN, EPI_NONE, torch.float32, False, False),
]


def main():
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    iters = int(os.environ.get("GEMM_ITERS", "20"))
    rows = []
    for name, M, N, Kd, am, bm, epi, odt, aux, bias in SHAPES:
        A = torch.randn((M, Kd) if am == MAJOR_K else (Kd, M), device=dev).bfloat16()
        B = torch.randn((N, Kd) if bm == MAJOR_K else (Kd, N), device=dev).bfloat16()
        kw = {}
        if bias:
            kw["bias"] = torch.randn(N, device=dev)
        if epi == EPI_SCALE_RESIDUAL:
            kw["gamma"] = torch.randn(N, device=dev)
            kw["residual"] = torch.randn(M, N, device=dev)
        if epi == EPI_DGELU:
            kw["aux"] = torch.randn(M, N, device=dev).bfloat16()
        elif aux:
            kw["want_aux_dtype"] = torch.bfloat16
        out = torch.empty(M, N, dtype=odt, device=dev)

        def run():
            K.gemm(BF16, A, am, B, bm, M, N, Kd, odt, epilogue=epi, out=out, **kw)
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            run()
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) / iters * 1e3
        # correctness spot check against fp32 math on a slab of rows
        rs = slice(0, 256)
        Af = (A[rs] if am == MAJOR_K else A[:, rs].t()).float()
        Bf = (B if bm == MAJOR_K else B.t()).float()
        ref = Af @ Bf.t()
        if bias:
            ref = ref + kw["bias"]
        if epi == EPI_GELU:
            ref = torch.nn.functional.gelu(ref)
        elif epi == EPI_SCALE_RESIDUAL:
            ref = kw["residual"][rs] + kw["gamma"] * ref
        elif epi == EPI_DGELU:
            h = kw["aux"][rs].float().requires_grad_(True)
            (dg,) = torch.autograd.grad(torch.nn.functional.gelu(h), h, torch.ones_like(h))
            ref = ref * dg
        err = float((out[rs].float() - ref).abs().max() / ref.abs().max())
        row = dict(shape=name, M=M, N=N, K=Kd, us=round(us, 1), tflops=round(2.0 * M * N * Kd / us / 1e6, 1), relerr=round(err, 5))
        rows.append(row)
        print(json.dumps(row), flush=True)
    tot = sum(r["us"] for r in rows)
    print(json.dumps(dict(total_us=round(tot, 1))), flush=True)


if __name__ == "__main__":
    main()
