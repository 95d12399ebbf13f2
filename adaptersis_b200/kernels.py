"""Tensor-level wrappers over the C ABI (no autograd here).  Each function allocates its outputs
with torch (device memory is PyTorch's job), passes raw pointers + sizes + the current CUDA stream
to libasis_b200.so and returns.  Argument order follows include/asis_b200.h."""
import ctypes

import torch

from . import _lib
from ._lib import (BF16, EPI_ACCUMULATE, EPI_DGELU, EPI_GELU, EPI_GELU_GRAD, EPI_MUL_AUX, EPI_NONE, EPI_SCALE_RESIDUAL,
                   F32, MAJOR_K, MAJOR_MN, check, dt, need_cuda, ptr, stream, workspace)

TORCH_DT = {F32: torch.float32, BF16: torch.bfloat16}

# optional per-launch profiler (bench.py): an object with .begin(name, work, unit) -> token and
# .end(token); records CUDA events on the launching stream around the kernel(s) of one op
_PROF = [None]


def set_profiler(p):
    _PROF[0] = p


class _Span:
    __slots__ = ("tok",)

    def __init__(self, name, work, unit, detail=None):
        p = _PROF[0]
        self.tok = p.begin(name, work, unit, detail) if p is not None else None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        if self.tok is not None:
            _PROF[0].end(self.tok)
        return False


def _c(t):
    return t if t.is_contiguous() else t.contiguous()


# ------------------------------------------------------------------------------------------ MSDA
def msda_forward(value, spatial_shapes, level_start_index, sampling_locations, attention_weights):
    need_cuda(value, spatial_shapes, level_start_index, sampling_locations, attention_weights)
    N, S, M, D = value.shape
    _, Lq, _, L, P, _ = sampling_locations.shape
    value = _c(value)
    loc = _c(sampling_locations.float())
    aw = _c(attention_weights.float())
    ss = _c(spatial_shapes.to(torch.int64))
    lsi = _c(level_start_index.to(torch.int64))
    out = torch.empty(N, Lq, M * D, dtype=value.dtype, device=value.device)
    e = value.element_size()
    pts = N * Lq * M * L * P
    with _Span("msda_fwd", e * N * S * M * D + 12 * pts + e * N * Lq * M * D, "B"):
        check(_lib.load().asis_msda_forward(ptr(value), dt(value), ptr(ss), ptr(lsi), ptr(loc), ptr(aw), ptr(out),
                                            dt(out), N, S, M, D, Lq, L, P, stream()))
    return out


def msda_backward(value, spatial_shapes, level_start_index, sampling_locations, attention_weights, grad_out):
    need_cuda(value, grad_out)
    N, S, M, D = value.shape
    _, Lq, _, L, P, _ = sampling_locations.shape
    lib = _lib.load()
    value = _c(value)
    loc = _c(sampling_locations.float())
    aw = _c(attention_weights.float())
    ss = _c(spatial_shapes.to(torch.int64))
    lsi = _c(level_start_index.to(torch.int64))
    grad_out = _c(grad_out.to(value.dtype))
    gv = torch.empty_like(value)
    gl = torch.empty_like(loc)
    ga = torch.empty_like(aw)
    nbytes = lib.asis_msda_backward_workspace_bytes(N, S, M, D, Lq, L, P)
    ws = workspace(nbytes, value.device)
    e = value.element_size()
    pts = N * Lq * M * L * P
    with _Span("msda_bwd", e * N * Lq * M * D + 2 * e * N * S * M * D + 24 * pts, "B"):
        check(lib.asis_msda_backward(ptr(value), dt(value), ptr(ss), ptr(lsi), ptr(loc), ptr(aw), ptr(grad_out),
                                     dt(grad_out), ptr(gv), ptr(gl), ptr(ga), N, S, M, D, Lq, L, P, ptr(ws), nbytes,
                                     stream()))
    return gv, gl, ga


def _ref_layout(reference_points, R, Lq, L):
    ref = _c(reference_points.float())
    rows = ref.shape[0] * ref.shape[1]
    if rows not in (R, Lq):
        raise RuntimeError(f"reference_points rows {tuple(reference_points.shape)} do not match queries")
    return ref, rows, ref.shape[2], ref.shape[3]


def msda_prep_forward(offsets, logits, reference_points, spatial_shapes, N, Lq, M, L, P):
    """offsets [N,Lq,M*L*P*2], logits [N,Lq,M*L*P] -> loc [N,Lq,M,L,P,2], attn [N,Lq,M,L,P] (f32)."""
    need_cuda(offsets, logits, reference_points)
    R = N * Lq
    if reference_points.shape[-1] not in (2, 4):
        raise ValueError(
            "Last dim of reference_points must be 2 or 4, but get {} instead.".format(reference_points.shape[-1]))
    ref, rows, rl, rd = _ref_layout(reference_points, R, Lq, L)
    offsets = _c(offsets)
    logits = _c(logits.to(offsets.dtype))
    ss = _c(spatial_shapes.to(torch.int64))
    loc = torch.empty(N, Lq, M, L, P, 2, dtype=torch.float32, device=offsets.device)
    attn = torch.empty(N, Lq, M, L, P, dtype=torch.float32, device=offsets.device)
    check(_lib.load().asis_msda_prep_forward(ptr(offsets), ptr(logits), dt(offsets), ptr(ref), rows, rl, rd,
                                             ptr(ss), ptr(loc), ptr(attn), R, Lq, M, L, P, stream()))
    return loc, attn


def msda_prep_backward(grad_loc, grad_attn, attn, reference_points, spatial_shapes, out_dtype, N, Lq, M, L, P):
    R = N * Lq
    ref, rows, rl, rd = _ref_layout(reference_points, R, Lq, L)
    ss = _c(spatial_shapes.to(torch.int64))
    goff = torch.empty(N, Lq, M * L * P * 2, dtype=out_dtype, device=attn.device)
    glog = torch.empty(N, Lq, M * L * P, dtype=out_dtype, device=attn.device)
    check(_lib.load().asis_msda_prep_backward(ptr(_c(grad_loc)), ptr(_c(grad_attn)), ptr(attn), ptr(ref), rows, rl,
                                              rd, ptr(ss), ptr(goff), ptr(glog), dt(goff), R, Lq, M, L, P,
                                              stream()))
    return goff, glog


# ------------------------------------------------------------------------------------- LayerNorm
def layernorm_forward(x2d, weight, bias, eps, out_dtype):
    need_cuda(x2d, weight, bias)
    R, C = x2d.shape
    x2d = _c(x2d)
    y = torch.empty(R, C, dtype=out_dtype, device=x2d.device)
    mean = torch.empty(R, dtype=torch.float32, device=x2d.device)
    rstd = torch.empty(R, dtype=torch.float32, device=x2d.device)
    with _Span("ln_fwd", R * C * (x2d.element_size() + y.element_size()), "B"):
        check(_lib.load().asis_layernorm_forward(ptr(x2d), dt(x2d), ptr(weight), ptr(bias), ptr(y), dt(y),
                                                 ptr(mean), ptr(rstd), R, C, float(eps), stream()))
    return y, mean, rstd


def layernorm_backward(dy2d, x2d, weight, mean, rstd, dres=None, want_param_grads=True):
    """dx (f32) = dres + LN'(dy); returns dx, dweight, dbias (f32 or None)."""
    R, C = x2d.shape
    lib = _lib.load()
    dy2d = _c(dy2d)
    dx = torch.empty(R, C, dtype=torch.float32, device=x2d.device)
    dw = torch.empty(C, dtype=torch.float32, device=x2d.device) if want_param_grads else None
    db = torch.empty(C, dtype=torch.float32, device=x2d.device) if want_param_grads else None
    nbytes = lib.asis_layernorm_backward_workspace_bytes(R, C)
    ws = workspace(nbytes, x2d.device)
    if dres is not None:
        dres = _c(dres.float())
    nb = R * C * (dy2d.element_size() + x2d.element_size() + 4 + (4 if dres is not None else 0))
    with _Span("ln_bwd", nb, "B"):
        check(lib.asis_layernorm_backward(ptr(dy2d), dt(dy2d), ptr(x2d), dt(x2d), ptr(weight), ptr(mean), ptr(rstd),
                                          ptr(dres), ptr(dx), ptr(dw), ptr(db), 0, R, C, ptr(ws), nbytes, stream()))
    return dx, dw, db


# ------------------------------------------------------------------------------------------ GEMM
def gemm(compute, A, a_major, B, b_major, M, N, K, out_dtype, epilogue=EPI_NONE, bias=None, gamma=None,
         residual=None, aux=None, out=None, want_aux_dtype=None):
    """C[M,N] = epi(sum_k A[m,k] B[n,k]).  A/B are 2-D row-major tensors whose contiguous dimension
    is K (major K) or the M/N dimension (major MN).  Returns (C, aux)."""
    need_cuda(A, B)
    A = _c(A)
    B = _c(B)
    dev = A.device
    if out is None:
        out = torch.empty(M, N, dtype=out_dtype, device=dev)
    if epilogue in (EPI_GELU, EPI_SCALE_RESIDUAL, EPI_GELU_GRAD) and aux is None and want_aux_dtype is not None:
        aux = torch.empty(M, N, dtype=want_aux_dtype, device=dev)
    if residual is not None:
        assert residual.dtype == torch.float32 and residual.shape[-1] == N
        # the kernels read the residual with C's row pitch (ldc): a residual laid out like `out` is passed as it is
        if residual.dim() != 2 or residual.stride() != (out.stride(0), 1):
            if out.stride(0) != N:
                raise ValueError(f"gemm: the residual must have out's row pitch {out.stride(0)} (strides {residual.stride()})")
            residual = residual.contiguous()
    detail = None
    if _PROF[0] is not None:
        detail = (f"M={M} N={N} K={K} {'KM'[a_major]}/{'KM'[b_major]} epi={epilogue} out={'bf16' if out.dtype == torch.bfloat16 else 'f32'}"
                  f"{' aux' if aux is not None else ''}{' bias' if bias is not None else ''}")
    with _Span("gemm_bf16" if compute == BF16 else "gemm_f32", 2.0 * M * N * K, "FLOP", detail):
        check(_lib.load().asis_gemm(compute, ptr(A), a_major, A.stride(0), ptr(B), b_major, B.stride(0), ptr(out),
                                    dt(out), out.stride(0), M, N, K, epilogue, ptr(bias), ptr(gamma), ptr(residual),
                                    ptr(aux), dt(aux) if aux is not None else 0,
                                    aux.stride(0) if aux is not None else 0, stream()))
    return out, aux


def colsum(X2d, Y2d=None, out=None, accumulate=False):
    need_cuda(X2d)
    M, N = X2d.shape
    lib = _lib.load()
    X2d = _c(X2d)
    if Y2d is not None:
        Y2d = _c(Y2d)
    if out is None:
        out = torch.empty(N, dtype=torch.float32, device=X2d.device)
    nbytes = lib.asis_colsum_workspace_bytes(M, N)
    ws = workspace(nbytes, X2d.device)
    nb = M * N * (X2d.element_size() + (Y2d.element_size() if Y2d is not None else 0))
    with _Span("colsum", nb, "B"):
        check(lib.asis_colsum(ptr(X2d), dt(X2d), ptr(Y2d), dt(Y2d) if Y2d is not None else 0, X2d.stride(0),
                              ptr(out), int(accumulate), M, N, ptr(ws), nbytes, stream()))
    return out


def scale_cols(a2d, gamma, out_dtype):
    M, N = a2d.shape
    a2d = _c(a2d)
    out = torch.empty(M, N, dtype=out_dtype, device=a2d.device)
    with _Span("scale_cols", M * N * (a2d.element_size() + out.element_size()), "B"):
        check(_lib.load().asis_scale_cols(ptr(a2d), dt(a2d), ptr(gamma), ptr(out), dt(out), M, N, stream()))
    return out


def layerscale_backward(d2d, u2d, gamma, out_dtype, want_dgamma, want_dbias):
    """d [M, N] f32 -> du = d * gamma (out_dtype), dgamma = colsum(d * u), dbias = colsum(du) (f32 or None)."""
    M, N = d2d.shape
    lib = _lib.load()
    d2d = _c(d2d)
    dev = d2d.device
    du = torch.empty(M, N, dtype=out_dtype, device=dev)
    dgamma = torch.empty(N, dtype=torch.float32, device=dev) if want_dgamma else None
    dbias = torch.empty(N, dtype=torch.float32, device=dev) if want_dbias else None
    u = _c(u2d) if (want_dgamma and u2d is not None) else None
    assert u is None or u.dtype == out_dtype
    nbytes = lib.asis_layerscale_backward_workspace_bytes(M, N)
    ws = workspace(nbytes, dev)
    nb = M * N * (4 + du.element_size() + (u.element_size() if u is not None else 0))
    with _Span("layerscale_bwd", nb, "B"):
        check(lib.asis_layerscale_backward(ptr(d2d), ptr(u), ptr(gamma), ptr(du), dt(du), ptr(dgamma), ptr(dbias), M, N,
                                           ptr(ws), nbytes, stream()))
    return du, dgamma, dbias


def add(a, b, out_dtype):
    a = _c(a)
    b = _c(b)
    out = torch.empty(a.shape, dtype=out_dtype, device=a.device)
    check(_lib.load().asis_add(ptr(a), dt(a), ptr(b), dt(b), ptr(out), dt(out), a.numel(), stream()))
    return out


def cast(a, out_dtype):
    if a.dtype == out_dtype:
        return a
    a = _c(a)
    out = torch.empty(a.shape, dtype=out_dtype, device=a.device)
    check(_lib.load().asis_cast(ptr(a), dt(a), ptr(out), dt(out), a.numel(), stream()))
    return out


# ------------------------------------------------------------------------------------- attention
def attention_forward(compute, qkv, B, T, H, hd):
    """qkv [B,T,3*H*hd] (packed [3,H,hd]) -> out [B,T,H*hd], lse [B,H,T]."""
    need_cuda(qkv)
    lib = _lib.load()
    qkv = _c(qkv)
    out = torch.empty(B, T, H * hd, dtype=qkv.dtype, device=qkv.device)
    lse = torch.empty(B, H, T, dtype=torch.float32, device=qkv.device)
    nbytes = lib.asis_attention_forward_workspace_bytes(compute, B, T, H, hd)
    ws = workspace(nbytes, qkv.device)
    with _Span("attn_fwd", 4.0 * B * H * T * T * hd, "FLOP"):
        check(lib.asis_attention_forward(compute, ptr(qkv), ptr(out), ptr(lse), B, T, H, hd, ptr(ws), nbytes,
                                         stream()))
    return out, lse


def attention_backward(compute, qkv, out, lse, dout, B, T, H, hd):
    lib = _lib.load()
    dout = _c(dout.to(qkv.dtype))
    dqkv = torch.empty_like(qkv)
    nbytes = lib.asis_attention_backward_workspace_bytes(compute, B, T, H, hd)
    ws = workspace(nbytes, qkv.device)
    with _Span("attn_bwd", 10.0 * B * H * T * T * hd, "FLOP"):   # algorithmic: 5 GEMMs (7 are executed)
        check(lib.asis_attention_backward(compute, ptr(qkv), ptr(out), ptr(lse), ptr(dout), ptr(dqkv), B, T, H, hd,
                                          ptr(ws), nbytes, stream()))
    return dqkv


# ---------------------------------------------------------------------------------- front / conv
def patchify(img, patch, out_dtype, ldk):
    need_cuda(img)
    B, Cin, H, W = img.shape
    if H % patch != 0:
        raise AssertionError(f"Input image height {H} is not a multiple of patch height {patch}")
    if W % patch != 0:
        raise AssertionError(f"Input image width {W} is not a multiple of patch width: {patch}")
    img = _c(img.float())
    cols = torch.empty(B * (H // patch) * (W // patch), ldk, dtype=out_dtype, device=img.device)
    check(_lib.load().asis_patchify(ptr(img), ptr(cols), dt(cols), B, Cin, H, W, patch, ldk, stream()))
    return cols


def _int_array(vals):
    return (ctypes.c_int * len(vals))(*vals)


def dwconv3x3_forward(x, weight, bias, maps, fuse_gelu, save_pre):
    """x [B, n_tok, C]; maps = [(h, w), ...] back to back along n_tok."""
    need_cuda(x, weight, bias)
    B, ntok, C = x.shape
    assert sum(h * w for h, w in maps) == ntok
    x = _c(x)
    y = torch.empty_like(x)
    pre = torch.empty_like(x) if (fuse_gelu and save_pre) else None
    hs = _int_array([h for h, _ in maps])
    ws_ = _int_array([w for _, w in maps])
    check(_lib.load().asis_dwconv3x3_forward(ptr(x), dt(x), ptr(_c(weight.float())), ptr(_c(bias.float())), ptr(pre),
                                             ptr(y), B, C, len(maps), hs, ws_, int(fuse_gelu), stream()))
    return y, pre


def dwconv3x3_backward(dy, pre, x, weight, maps, fuse_gelu):
    B, ntok, C = x.shape
    lib = _lib.load()
    dy = _c(dy.to(x.dtype))
    dx = torch.empty_like(x)
    dw = torch.empty(C, 1, 3, 3, dtype=torch.float32, device=x.device)
    db = torch.empty(C, dtype=torch.float32, device=x.device)
    hs = _int_array([h for h, _ in maps])
    ws_ = _int_array([w for _, w in maps])
    nbytes = lib.asis_dwconv3x3_backward_workspace_bytes(B, C, ntok)
    ws = workspace(nbytes, x.device)
    check(lib.asis_dwconv3x3_backward(ptr(dy), ptr(pre), ptr(x), dt(x), ptr(_c(weight.float())), ptr(dx), ptr(dw),
                                      ptr(db), 0, B, C, len(maps), hs, ws_, int(fuse_gelu), ptr(ws), nbytes,
                                      stream()))
    return dx, dw, db


# ------------------------------------------------------------------------------------------ optimizer
def sgd_step(params, grads, bufs, lr, momentum, weight_decay):
    """torch.optim.SGD(momentum, weight_decay) update of a list of contiguous f32 tensors in place (asis_sgd_step)."""
    import ctypes
    n = len(params)
    if n == 0:
        return
    for t in (*params, *grads, *bufs):
        assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()
    P = (ctypes.c_void_p * n)(*[t.data_ptr() for t in params])
    G = (ctypes.c_void_p * n)(*[t.data_ptr() for t in grads])
    M = (ctypes.c_void_p * n)(*[t.data_ptr() for t in bufs])
    N = (ctypes.c_int64 * n)(*[t.numel() for t in params])
    check(_lib.load().asis_sgd_step(n, P, G, M, N, float(lr), float(momentum), float(weight_decay), stream()))


# ------------------------------------------------------------------------------------------ input ingest
def frames_to_batch(frames_u8, masks_u8=None, img_out=None, target_out=None):
    """frames [B, H, W, 3] uint8 (device) -> img [B, 3, H, W] f32 = frames / 255; masks [B, H, W] uint8 -> target int64
    (tools/dataset.py:111-118 on the device).  ``img_out`` / ``target_out``: write into existing buffers (the captured
    step's static inputs)."""
    need_cuda(frames_u8)
    B, H, W, C = frames_u8.shape
    assert C == 3 and frames_u8.dtype == torch.uint8 and frames_u8.is_contiguous()
    img = img_out if img_out is not None else torch.empty(B, 3, H, W, dtype=torch.float32, device=frames_u8.device)
    assert img.shape == (B, 3, H, W) and img.dtype == torch.float32 and img.is_contiguous()
    tgt = None
    if masks_u8 is not None:
        assert masks_u8.shape == (B, H, W) and masks_u8.dtype == torch.uint8 and masks_u8.is_contiguous()
        tgt = target_out if target_out is not None else torch.empty(B, H, W, dtype=torch.int64, device=frames_u8.device)
        assert tgt.shape == (B, H, W) and tgt.dtype == torch.int64 and tgt.is_contiguous()
    check(_lib.load().asis_frames_to_batch(ptr(frames_u8), ptr(img), ptr(masks_u8), ptr(tgt), B, H, W, stream()))
    return img, tgt


# ------------------------------------------------------------------------------------------ decoder
def upsample2x_forward(x_nhwc, pad_in=0, pad_out=0):
    """x [B, H(+2pi), W(+2pi), C] contiguous -> [B, 2H(+2po), 2W(+2po), C]; bilinear, align_corners=True."""
    need_cuda(x_nhwc)
    B, Hs, Ws, C = x_nhwc.shape
    H, W = Hs - 2 * pad_in, Ws - 2 * pad_in
    y = torch.empty(B, 2 * H + 2 * pad_out, 2 * W + 2 * pad_out, C, dtype=x_nhwc.dtype, device=x_nhwc.device)
    nb = x_nhwc.element_size() * B * H * W * C * 5
    with _Span("upsample2x_fwd", nb, "B"):
        check(_lib.load().asis_upsample2x_bilinear_forward_padded(ptr(x_nhwc), ptr(y), dt(x_nhwc), B, H, W, C, pad_in, pad_out,
                                                                  stream()))
    return y


def upsample2x_backward(gy_nhwc, pad_in=0, pad_out=0):
    """gy [B, 2H(+2po), 2W(+2po), C] contiguous -> gx [B, H(+2pi), W(+2pi), C]."""
    need_cuda(gy_nhwc)
    B, OHs, OWs, C = gy_nhwc.shape
    H, W = (OHs - 2 * pad_out) // 2, (OWs - 2 * pad_out) // 2
    gx = torch.empty(B, H + 2 * pad_in, W + 2 * pad_in, C, dtype=gy_nhwc.dtype, device=gy_nhwc.device)
    nb = gy_nhwc.element_size() * B * H * W * C * 5
    with _Span("upsample2x_bwd", nb, "B"):
        check(_lib.load().asis_upsample2x_bilinear_backward_padded(ptr(gy_nhwc), ptr(gx), dt(gy_nhwc), B, H, W, C, pad_in, pad_out,
                                                                   stream()))
    return gx


# ------------------------------------------------------------------- convolutional stages (SPM, decoder)
def conv_out_size(n, k, stride, pad):
    return (n + 2 * pad - k) // stride + 1


def im2col(x, k, stride, pad, out_dtype, storage_pad=0):
    """x [B, H+2sp, W+2sp, C] channels-last -> cols [B*Ho*Wo, ldk], K = (ky, kx, c), ldk = k*k*C rounded up to 8."""
    need_cuda(x)
    B, Hs, Ws, C = x.shape
    H, W = Hs - 2 * storage_pad, Ws - 2 * storage_pad
    Ho, Wo = conv_out_size(H, k, stride, pad), conv_out_size(W, k, stride, pad)
    Kd = k * k * C
    ldk = (Kd + 7) // 8 * 8
    x = _c(x)
    cols = torch.empty(B * Ho * Wo, ldk, dtype=out_dtype, device=x.device)
    nb = cols.numel() * cols.element_size() + B * H * W * C * x.element_size()
    with _Span("im2col", nb, "B"):
        check(_lib.load().asis_im2col(ptr(x), dt(x), ptr(cols), dt(cols), B, H, W, C, storage_pad, k, stride, pad, ldk,
                                      stream()))
    return cols, (Ho, Wo)


def col2im(dcols, B, H, W, C, k, stride, pad, storage_pad=0):
    """dcols [B*Ho*Wo, ldk] -> dx [B, H+2sp, W+2sp, C] (gather over the taps that touch an input pixel)."""
    need_cuda(dcols)
    dcols = _c(dcols)
    dx = torch.empty(B, H + 2 * storage_pad, W + 2 * storage_pad, C, dtype=dcols.dtype, device=dcols.device)
    nb = (dcols.numel() + dx.numel()) * dcols.element_size()
    with _Span("col2im", nb, "B"):
        check(_lib.load().asis_col2im(ptr(dcols), ptr(dx), dt(dx), B, H, W, C, storage_pad, k, stride, pad,
                                      dcols.stride(0), stream()))
    return dx


def chan_stats(x, shift, storage_pad=0):
    """x [B, Hs, Ws, C] -> s [2, C] f32: sum (x - shift), sum (x - shift)^2 over the logical pixels."""
    need_cuda(x, shift)
    lib = _lib.load()
    B, Hs, Ws, C = x.shape
    H, W = Hs - 2 * storage_pad, Ws - 2 * storage_pad
    x = _c(x)
    s = torch.empty(2, C, dtype=torch.float32, device=x.device)
    nbytes = lib.asis_chan_stats_workspace_bytes(B, H, W, C)
    ws = workspace(nbytes, x.device)
    with _Span("bn_stats", x.numel() * x.element_size(), "B"):
        check(lib.asis_chan_stats(0, ptr(x), None, dt(x), B, H, W, C, storage_pad, 0, ptr(shift), None, None, None, None, 0,
                                  ptr(s), ptr(s[1]), ptr(ws), nbytes, stream()))
    return s


def chan_stats_backward(x, dy, a, b, mean, rstd, relu, storage_pad=0, dy_pad=0):
    """-> s [2, C] f32: sum dz, sum dz * xhat  (dz = dy * relu'(a (x - mean) + b)); x / dy may use different storage padding."""
    lib = _lib.load()
    B, Hs, Ws, C = x.shape
    H, W = Hs - 2 * storage_pad, Ws - 2 * storage_pad
    x, dy = _c(x), _c(dy)
    assert dy.dtype == x.dtype and dy.shape == (B, H + 2 * dy_pad, W + 2 * dy_pad, C)
    s = torch.empty(2, C, dtype=torch.float32, device=x.device)
    nbytes = lib.asis_chan_stats_workspace_bytes(B, H, W, C)
    ws = workspace(nbytes, x.device)
    with _Span("bn_bwd_stats", 2 * x.numel() * x.element_size(), "B"):
        check(lib.asis_chan_stats(1, ptr(x), ptr(dy), dt(x), B, H, W, C, storage_pad, dy_pad, None, ptr(a), ptr(b), ptr(mean),
                                  ptr(rstd), int(relu), ptr(s), ptr(s[1]), ptr(ws), nbytes, stream()))
    return s


def bn_apply(x, a, b, mean, relu, out_dtype, pad_in=0, pad_out=0):
    """y = act(a[c] (x - mean[c]) + b[c]) on a channels-last map (optionally re-padding the storage)."""
    need_cuda(x, a, b, mean)
    B, Hs, Ws, C = x.shape
    H, W = Hs - 2 * pad_in, Ws - 2 * pad_in
    x = _c(x)
    y = torch.empty(B, H + 2 * pad_out, W + 2 * pad_out, C, dtype=out_dtype, device=x.device)
    with _Span("bn_apply", x.numel() * x.element_size() + y.numel() * y.element_size(), "B"):
        check(_lib.load().asis_bn_apply(0, ptr(x), None, dt(x), ptr(y), dt(y), B, H, W, C, pad_in, pad_out, 0, ptr(a), ptr(b),
                                        ptr(mean), None, None, None, int(relu), stream()))
    return y


def bn_apply_backward(x, dy, a, b, mean, rstd, c1, c2, relu, pad=0, dy_pad=0):
    """dx = a * (dz - c1 - xhat * c2), in x's storage (zero border); dy in storage dy_pad."""
    B, Hs, Ws, C = x.shape
    H, W = Hs - 2 * pad, Ws - 2 * pad
    x, dy = _c(x), _c(dy)
    dx = torch.empty_like(x)
    with _Span("bn_bwd_apply", 3 * x.numel() * x.element_size(), "B"):
        check(_lib.load().asis_bn_apply(1, ptr(x), ptr(dy), dt(x), ptr(dx), dt(dx), B, H, W, C, pad, pad, dy_pad, ptr(a), ptr(b),
                                        ptr(mean), ptr(rstd), ptr(c1), ptr(c2), int(relu), stream()))
    return dx


def maxpool3x3s2_forward(x):
    need_cuda(x)
    B, H, W, C = x.shape
    x = _c(x)
    Ho, Wo = conv_out_size(H, 3, 2, 1), conv_out_size(W, 3, 2, 1)
    y = torch.empty(B, Ho, Wo, C, dtype=x.dtype, device=x.device)
    idx = torch.empty(B, Ho, Wo, C, dtype=torch.uint8, device=x.device)
    check(_lib.load().asis_maxpool3x3s2_forward(ptr(x), ptr(y), ptr(idx), dt(x), B, H, W, C, 0, 0, stream()))
    return y, idx


def maxpool3x3s2_backward(gy, idx, H, W):
    B, Ho, Wo, C = gy.shape
    gy = _c(gy)
    gx = torch.empty(B, H, W, C, dtype=gy.dtype, device=gy.device)
    check(_lib.load().asis_maxpool3x3s2_backward(ptr(gy), ptr(idx), ptr(gx), dt(gy), B, H, W, C, 0, 0, stream()))
    return gx


def seg_head_forward(z, w2, bias, CO):
    """conv3x3_pad1(upsample2x(z)) + bias, fused: z [B,H,W,C] channels-last, w2 [9*CO, C] f32 -> y [B,2H,2W,CO] f32."""
    need_cuda(z, w2)
    lib = _lib.load()
    B, H, W, C = z.shape
    z = _c(z)
    y = torch.empty(B, 2 * H, 2 * W, CO, dtype=torch.float32, device=z.device)
    nbytes = lib.asis_seg_head_workspace_bytes(B, H, W, C, CO)
    ws = workspace(nbytes, z.device)
    with _Span("seg_head_fwd", z.numel() * z.element_size() + y.numel() * 4, "B"):
        check(lib.asis_seg_head_forward(ptr(z), dt(z), ptr(w2), ptr(bias), ptr(y), B, H, W, C, CO, ptr(ws), nbytes, stream()))
    return y


def seg_head_backward(z, w2, gy, need_gz, need_gw):
    lib = _lib.load()
    B, H, W, C = z.shape
    CO = gy.shape[-1]
    z, gy = _c(z), _c(gy.float())
    gz = torch.empty_like(z) if need_gz else None
    gw2 = torch.empty(9 * CO, C, dtype=torch.float32, device=z.device) if need_gw else None
    nbytes = lib.asis_seg_head_workspace_bytes(B, H, W, C, CO)
    ws = workspace(nbytes, z.device)
    with _Span("seg_head_bwd", 2 * z.numel() * z.element_size() + gy.numel() * 4, "B"):
        check(lib.asis_seg_head_backward(ptr(z), dt(z), ptr(w2), ptr(gy), ptr(gz), ptr(gw2), B, H, W, C, CO, ptr(ws), nbytes,
                                         stream()))
    return gz, gw2


def conv3x3s1_gemm(op, a, b, out, bias, B, H, W, Cin, Cout):
    """Implicit-GEMM pieces of a 3x3 / stride 1 / pad 1 convolution over zero-padded channels-last bf16 maps
    (include/asis_b200.h: asis_conv3x3s1_gemm).  `out` is allocated by the caller."""
    need_cuda(a, b, out)
    flops = 2.0 * B * (H + 2) * (W + 2) * 9 * Cin * Cout
    with _Span("conv_bf16", flops, "FLOP", f"conv3x3 op={op} B={B} {H}x{W} Cin={Cin} Cout={Cout}" if _PROF[0] is not None else None):
        check(_lib.load().asis_conv3x3s1_gemm(op, ptr(a), ptr(b), ptr(out), dt(out), ptr(bias), B, H, W, Cin, Cout, stream()))
    return out
