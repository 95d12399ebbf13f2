"""Diagnostics for the tcgen05 kernels: prints max-relative errors per variant instead of asserting,
one group per process invocation (so that a hang in one group cannot hide the others)."""
import sys
import os
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from adaptersis_b200 import kernels as K  # noqa: E402
from adaptersis_b200._lib import (BF16, EPI_ACCUMULATE, EPI_DGELU, EPI_GELU, EPI_NONE, EPI_SCALE_RESIDUAL,  # noqa: E402
                                  MAJOR_K, MAJOR_MN)

dev = "cuda"


def rel(a, b):
    a = a.double()
    b = b.double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def gemm_case(M, N, Kd, am, bm, tag):
    torch.manual_seed(0)
    A = torch.randn(M, Kd, device=dev).bfloat16()
    B = torch.randn(N, Kd, device=dev).bfloat16()
    ref = A.float() @ B.float().t()
    a = A if am == MAJOR_K else A.t().contiguous()
    b = B if bm == MAJOR_K else B.t().contiguous()
    c, _ = K.gemm(BF16, a, am, b, bm, M, N, Kd, torch.float32)
    torch.cuda.synchronize()
    print(f"gemm {tag} M={M} N={N} K={Kd}: rel err {rel(c, ref):.3e}", flush=True)


def main(group):
    if group == "gemm_kk":
        for shp in [(128, 256, 64), (128, 256, 256), (256, 512, 1024), (300, 200, 136), (1765, 1024, 1024), (21180, 3072, 1024)]:
            gemm_case(*shp, MAJOR_K, MAJOR_K, "K/K")
        M, N, Kd = 1000, 1024, 512
        A = torch.randn(M, Kd, device=dev).bfloat16()
        B = torch.randn(N, Kd, device=dev).bfloat16()
        ref = A.float() @ B.float().t()
        bias = torch.randn(N, device=dev)
        gamma = torch.randn(N, device=dev)
        res = torch.randn(M, N, device=dev)
        c, _ = K.gemm(BF16, A, MAJOR_K, B, MAJOR_K, M, N, Kd, torch.bfloat16, bias=bias)
        print("epi bias->bf16", rel(c.float(), ref + bias))
        c, aux = K.gemm(BF16, A, MAJOR_K, B, MAJOR_K, M, N, Kd, torch.bfloat16, epilogue=EPI_GELU, bias=bias, want_aux_dtype=torch.bfloat16)
        print("epi gelu", rel(c.float(), torch.nn.functional.gelu(ref + bias)), rel(aux.float(), ref + bias))
        c, aux = K.gemm(BF16, A, MAJOR_K, B, MAJOR_K, M, N, Kd, torch.float32, epilogue=EPI_SCALE_RESIDUAL, bias=bias, gamma=gamma, residual=res, want_aux_dtype=torch.bfloat16)
        print("epi scale_residual", rel(c, res + gamma * (ref + bias)), rel(aux.float(), ref + bias))
        h = torch.randn(M, N, device=dev, requires_grad=True)
        (dg,) = torch.autograd.grad(torch.nn.functional.gelu(h), h, torch.ones_like(h))
        c, _ = K.gemm(BF16, A, MAJOR_K, B, MAJOR_K, M, N, Kd, torch.bfloat16, epilogue=EPI_DGELU, aux=h.detach().bfloat16())
        (dg2,) = torch.autograd.grad(torch.nn.functional.gelu(h.detach().bfloat16().float().requires_grad_(True)), h, torch.ones_like(h), allow_unused=True) if False else (dg,)
        print("epi dgelu", rel(c.float(), ref * dg))
        acc = torch.randn(M, N, device=dev)
        want = acc + ref
        c, _ = K.gemm(BF16, A, MAJOR_K, B, MAJOR_K, M, N, Kd, torch.float32, epilogue=EPI_ACCUMULATE, out=acc)
        print("epi accumulate", rel(c, want))
    elif group == "gemm_kmn":
        for shp in [(128, 256, 64), (128, 256, 256), (300, 200, 136), (1765, 1024, 4096), (2000, 96, 1024), (2000, 1024, 192)]:
            gemm_case(*shp, MAJOR_K, MAJOR_MN, "K/MN")
    elif group == "gemm_mnmn":
        for shp in [(128, 256, 64), (128, 256, 256), (300, 200, 136), (1024, 1024, 21180), (4096, 1024, 3000), (192, 1024, 2000)]:
            gemm_case(*shp, MAJOR_MN, MAJOR_MN, "MN/MN")
        gemm_case(300, 200, 136, MAJOR_MN, MAJOR_K, "MN/K")
    elif group in ("attn_fwd", "attn_bwd"):
        for (B, T, H) in [(1, 128, 1), (1, 256, 2), (2, 300, 3), (1, 1765, 16)]:
            torch.manual_seed(1)
            C = H * 64
            qkv = torch.randn(B, T, 3 * C, device=dev).bfloat16()
            x = qkv.float().requires_grad_(True)
            q, k, v = x.view(B, T, 3, H, 64).permute(2, 0, 3, 1, 4)
            s = (q * 64 ** -0.5) @ k.transpose(-1, -2)
            p = torch.softmax(s, -1)
            ref = (p @ v).transpose(1, 2).reshape(B, T, C)
            lse_ref = torch.logsumexp(s, -1)
            out, lse = K.attention_forward(BF16, qkv, B, T, H, 64)
            torch.cuda.synchronize()
            print(f"attn fwd B={B} T={T} H={H}: out {rel(out.float(), ref):.3e} lse {rel(lse, lse_ref):.3e}", flush=True)
            if group == "attn_bwd":
                dout = torch.randn(B, T, C, device=dev).bfloat16()
                (g,) = torch.autograd.grad(ref, x, dout.float())
                dqkv = K.attention_backward(BF16, qkv, out, lse, dout, B, T, H, 64)
                torch.cuda.synchronize()
                gq, gk, gv = g.view(B, T, 3, C).unbind(2)
                dq, dk, dv = dqkv.float().view(B, T, 3, C).unbind(2)
                print(f"attn bwd B={B} T={T} H={H}: dq {rel(dq, gq):.3e} dk {rel(dk, gk):.3e} dv {rel(dv, gv):.3e}", flush=True)


def timeit(fn, iters=10):
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2]


def perf():
    R = 21180
    for tag, M, N, Kd, am, bm, odt in [
            ("qkv fwd K/K", R, 3072, 1024, MAJOR_K, MAJOR_K, torch.bfloat16),
            ("proj fwd K/K", R, 1024, 1024, MAJOR_K, MAJOR_K, torch.bfloat16),
            ("fc1 fwd K/K", R, 4096, 1024, MAJOR_K, MAJOR_K, torch.bfloat16),
            ("fc2 fwd K/K", R, 1024, 4096, MAJOR_K, MAJOR_K, torch.bfloat16),
            ("fc1 dgrad K/MN", R, 1024, 4096, MAJOR_K, MAJOR_MN, torch.bfloat16),
            ("fc2 dgrad K/MN", R, 4096, 1024, MAJOR_K, MAJOR_MN, torch.bfloat16),
            ("fc1 wgrad MN/MN", 4096, 1024, R, MAJOR_MN, MAJOR_MN, torch.float32),
            ("proj wgrad MN/MN", 1024, 1024, R, MAJOR_MN, MAJOR_MN, torch.float32),
            ("value_proj inj K/K", 12 * 6949, 1024, 1024, MAJOR_K, MAJOR_K, torch.bfloat16)]:
        a = torch.randn((M, Kd) if am == MAJOR_K else (Kd, M), device=dev).bfloat16()
        b = torch.randn((N, Kd) if bm == MAJOR_K else (Kd, N), device=dev).bfloat16()
        ms = timeit(lambda: K.gemm(BF16, a, am, b, bm, M, N, Kd, odt))
        print(f"gemm {tag:22s} M={M} N={N} K={Kd}: {ms * 1e3:8.1f} us  {2.0 * M * N * Kd / ms / 1e9:7.1f} TFLOP/s", flush=True)
    # fused epilogues on the fc1 / fc2 shapes
    A = torch.randn(R, 1024, device=dev).bfloat16()
    W1 = torch.randn(4096, 1024, device=dev).bfloat16()
    bias = torch.randn(4096, device=dev)
    ms = timeit(lambda: K.gemm(BF16, A, MAJOR_K, W1, MAJOR_K, R, 4096, 1024, torch.bfloat16, epilogue=EPI_GELU, bias=bias, want_aux_dtype=torch.bfloat16))
    print(f"gemm fc1+bias+GELU(+aux): {ms * 1e3:8.1f} us  {2.0 * R * 4096 * 1024 / ms / 1e9:7.1f} TFLOP/s", flush=True)
    ms = timeit(lambda: K.gemm(BF16, A, MAJOR_K, W1, MAJOR_K, R, 4096, 1024, torch.bfloat16, epilogue=EPI_GELU, bias=bias))
    print(f"gemm fc1+bias+GELU (no aux): {ms * 1e3:8.1f} us  {2.0 * R * 4096 * 1024 / ms / 1e9:7.1f} TFLOP/s", flush=True)
    ms = timeit(lambda: K.gemm(BF16, A, MAJOR_K, W1, MAJOR_K, R, 4096, 1024, torch.float32))
    print(f"gemm fc1 plain, fp32 out (2x store bytes): {ms * 1e3:8.1f} us  {2.0 * R * 4096 * 1024 / ms / 1e9:7.1f} TFLOP/s", flush=True)
    ms = timeit(lambda: K.gemm(BF16, A, MAJOR_K, W1, MAJOR_K, R, 4096, 1024, torch.bfloat16, bias=bias))
    print(f"gemm fc1+bias: {ms * 1e3:8.1f} us  {2.0 * R * 4096 * 1024 / ms / 1e9:7.1f} TFLOP/s", flush=True)
    G = torch.randn(R, 4096, device=dev).bfloat16()
    W2 = torch.randn(1024, 4096, device=dev).bfloat16()
    res = torch.randn(R, 1024, device=dev)
    gam = torch.randn(1024, device=dev)
    b2 = torch.randn(1024, device=dev)
    ms = timeit(lambda: K.gemm(BF16, G, MAJOR_K, W2, MAJOR_K, R, 1024, 4096, torch.float32, epilogue=EPI_SCALE_RESIDUAL, bias=b2, gamma=gam, residual=res, want_aux_dtype=torch.bfloat16))
    print(f"gemm fc2+bias+ls+residual(+aux): {ms * 1e3:8.1f} us  {2.0 * R * 4096 * 1024 / ms / 1e9:7.1f} TFLOP/s", flush=True)
    B, T, H = 12, 1765, 16
    qkv = torch.randn(B, T, 3 * H * 64, device=dev).bfloat16()
    ms = timeit(lambda: K.attention_forward(BF16, qkv, B, T, H, 64))
    print(f"attn fwd B={B} T={T} H={H}: {ms * 1e3:8.1f} us  {4.0 * B * H * T * T * 64 / ms / 1e9:7.1f} TFLOP/s", flush=True)
    out, lse = K.attention_forward(BF16, qkv, B, T, H, 64)
    dout = torch.randn_like(out)
    ms = timeit(lambda: K.attention_backward(BF16, qkv, out, lse, dout, B, T, H, 64))
    print(f"attn bwd: {ms * 1e3:8.1f} us  {10.0 * B * H * T * T * 64 / ms / 1e9:7.1f} TFLOP/s (algorithmic 5 GEMMs)", flush=True)
    x = torch.randn(R, 1024, device=dev)
    dy = torch.randn(R, 1024, device=dev).bfloat16()
    w = torch.randn(1024, device=dev)
    y, mean, rstd = K.layernorm_forward(x, w, w, 1e-6, torch.bfloat16)
    ms = timeit(lambda: K.layernorm_backward(dy, x, w, mean, rstd, x))
    print(f"ln_bwd R={R} C=1024: {ms * 1e3:8.1f} us  {R * 1024 * 14 / ms / 1e6:7.1f} GB/s", flush=True)
    ms = timeit(lambda: K.layernorm_forward(x, w, w, 1e-6, torch.bfloat16))
    print(f"ln_fwd: {ms * 1e3:8.1f} us  {R * 1024 * 6 / ms / 1e6:7.1f} GB/s", flush=True)
    big = torch.randn(R, 4096, device=dev).bfloat16()
    ms = timeit(lambda: K.colsum(big))
    print(f"colsum [R,4096] bf16: {ms * 1e3:8.1f} us  {R * 4096 * 2 / ms / 1e6:7.1f} GB/s", flush=True)


if __name__ == "__main__":
    if sys.argv[1] == "perf":
        perf()
        sys.exit(0)
    main(sys.argv[1])
