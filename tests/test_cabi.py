"""CPU-only checks of the drop-in boundary: the C-ABI library loads, exports every symbol that
include/asis_b200.h declares, validates arguments (no compute without a GPU), and the product
package has no CPU fallback."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "asis_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(asis_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from adaptersis_b200 import _lib
    lib = _lib.load()
    names = declared_symbols()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), f"libasis_b200.so does not export {n}"
    assert set(names) == set(_lib.SIGNATURES), set(names) ^ set(_lib.SIGNATURES)
    assert lib.asis_abi_version() == 1


def test_argument_validation_without_gpu():
    from adaptersis_b200 import _lib
    lib = _lib.load()
    rc = lib.asis_msda_forward(None, 0, None, None, None, None, None, 0, 1, 1, 1, 4, 1, 1, 1, None)
    assert rc == -1 and b"null pointer" in lib.asis_last_error()
    rc = lib.asis_msda_forward(None, 0, None, None, None, None, None, 0, 1, 1, 1, 6, 1, 1, 1, None)
    assert rc == -1 and b"multiple of 4" in lib.asis_last_error()
    rc = lib.asis_gemm(0, None, 0, 8, None, 0, 8, None, 0, 8, 8, 8, 8, 0, None, None, None, None, 0, 0, None)
    assert rc == -1
    assert lib.asis_msda_backward_workspace_bytes(2, 100, 4, 16, 10, 3, 4) >= 2 * 2 * 4 * 100 * 4 + 2 * 4 * 10 * 3 * 4 * 4 * 8
    assert lib.asis_attention_backward_workspace_bytes(0, 1, 10, 2, 16) == 2 * 2 * 100 * 4


def test_host_side_validation_and_workspace_sizes():
    """Host logic of the entry points added in round 1 (no kernel is launched: every call fails its
    argument check first, or only computes a size)."""
    import ctypes
    from adaptersis_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(256)          # a non-null, 16-byte aligned address that is never dereferenced
    # decoder resize: channel count must fill 16-byte vectors, H and W > 1
    rc = lib.asis_upsample2x_bilinear_forward(fake, fake, 1, 2, 8, 8, 12, None)
    assert rc == -1 and b"multiple of 8" in lib.asis_last_error()
    rc = lib.asis_upsample2x_bilinear_backward(fake, fake, 0, 2, 1, 8, 16, None)
    assert rc == -1 and b"H > 1" in lib.asis_last_error()
    rc = lib.asis_upsample2x_bilinear_forward(None, fake, 0, 2, 8, 8, 16, None)
    assert rc == -1 and b"null pointer" in lib.asis_last_error()
    # LayerScale backward: d gamma needs the saved branch output; workspace is checked before launch
    rc = lib.asis_layerscale_backward(fake, None, fake, fake, 1, fake, None, 64, 128, fake, 1 << 20, None)
    assert rc == -1 and b"needs the saved branch output" in lib.asis_last_error()
    need = lib.asis_layerscale_backward_workspace_bytes(21180, 1024)
    assert need >= 2 * 1024 * 4
    rc = lib.asis_layerscale_backward(fake, fake, fake, fake, 1, fake, fake, 21180, 1024, fake, need - 1, None)
    assert rc != 0 and b"workspace" in lib.asis_last_error()
    # MSDA backward workspace: cursor table (chunks x pixels) + pixel pointers + 8-byte entries; the
    # table is capped (256 MB) by using fewer, longer query chunks
    def ws(N, S, M, D, Lq, L, P):
        return lib.asis_msda_backward_workspace_bytes(N, S, M, D, Lq, L, P)
    entries = 12 * 8 * 1764 * 3 * 4 * 4 * 8
    w = ws(12, 6949, 8, 128, 1764, 3, 4)
    assert entries + 12 * 8 * 6949 * 4 <= w <= entries + 12 * 8 * 6949 * 4 * 8 + (1 << 20)
    assert ws(12, 6949, 8, 128, 3528, 3, 4) > w                      # more queries: more entries and chunks
    big = ws(12, 180000, 16, 8, 17000, 1, 4)
    assert big <= 12 * 16 * 17000 * 4 * 4 * 8 + (256 << 20) + 12 * 16 * 180001 * 4 + (1 << 20)
    assert ws(0, 10, 1, 8, 10, 1, 1) == 0
    # MSDA dimension limits are reported, not silently truncated
    rc = lib.asis_msda_forward(fake, 0, fake, fake, fake, fake, fake, 0, 1, 10, 1, 256, 5, 1, 1, None)
    assert rc == -1 and b"<= 128" in lib.asis_last_error()
    rc = lib.asis_msda_forward(fake, 0, fake, fake, fake, fake, fake, 0, 1, 10, 1, 8, 5, 9, 1, None)
    assert rc == -1 and b"n_levels" in lib.asis_last_error()


def test_host_side_validation_round2_entry_points():
    """The entry points added in round 2 (convolutional stages, optimizer, ingest): every call below fails its argument
    check before any CUDA call, or only computes a size."""
    import ctypes
    from adaptersis_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(256)
    # implicit 3x3 convolution: channels in 64s, op in {0, 1, 2}, f32 weight gradient
    rc = lib.asis_conv3x3s1_gemm(0, fake, fake, fake, 1, None, 2, 8, 8, 48, 64, None)
    assert rc == -1 and b"multiples of 64" in lib.asis_last_error()
    rc = lib.asis_conv3x3s1_gemm(3, fake, fake, fake, 1, None, 2, 8, 8, 64, 64, None)
    assert rc == -1 and b"op must be" in lib.asis_last_error()
    rc = lib.asis_conv3x3s1_gemm(2, fake, fake, fake, 1, None, 2, 8, 8, 64, 64, None)
    assert rc == -1 and b"weight gradient is f32" in lib.asis_last_error()
    rc = lib.asis_conv3x3s1_gemm(0, None, fake, fake, 1, None, 2, 8, 8, 64, 64, None)
    assert rc == -1 and b"null pointer" in lib.asis_last_error()
    # BatchNorm pieces: channel vectors, the one-buffer statistics layout, workspace before launch
    assert lib.asis_chan_stats_workspace_bytes(12, 294, 294, 64) >= 2 * 64 * 4
    s1 = ctypes.c_void_p(1024)
    rc = lib.asis_chan_stats(0, fake, None, 1, 2, 8, 8, 12, 0, 0, fake, None, None, None, None, 0, s1, ctypes.c_void_p(1024 + 48), fake, 1 << 20, None)
    assert rc == -1 and b"multiple of 8" in lib.asis_last_error()
    rc = lib.asis_chan_stats(0, fake, None, 1, 2, 8, 8, 16, 0, 0, fake, None, None, None, None, 0, s1, ctypes.c_void_p(4096), fake, 1 << 20, None)
    assert rc == -1 and b"s2 must follow s1" in lib.asis_last_error()
    rc = lib.asis_bn_apply(0, fake, None, 1, fake, 0, 2, 8, 8, 16, 0, 0, 0, fake, fake, fake, None, None, None, 1, None)
    assert rc == -1 and b"bf16 -> f32" in lib.asis_last_error()
    # segmentation head: 1..4 classes; workspace = low-resolution taps + weight-gradient partials
    assert lib.asis_seg_head_workspace_bytes(12, 336, 336, 64, 2) >= 12 * 336 * 336 * 18 * 4
    rc = lib.asis_seg_head_forward(fake, 1, fake, None, fake, 2, 8, 8, 64, 5, fake, 1 << 30, None)
    assert rc == -1 and b"1..4 classes" in lib.asis_last_error()
    rc = lib.asis_seg_head_forward(fake, 1, fake, None, fake, 2, 8, 8, 64, 2, fake, 16, None)
    assert rc != 0 and b"workspace" in lib.asis_last_error()
    # optimizer and ingest
    rc = lib.asis_sgd_step(3, None, None, None, None, 0.01, 0.99, 3e-5, None)
    assert rc == -1 and b"null table" in lib.asis_last_error()
    assert lib.asis_sgd_step(0, None, None, None, None, 0.01, 0.99, 3e-5, None) == 0            # nothing to do
    rc = lib.asis_frames_to_batch(fake, fake, fake, None, 2, 8, 8, None)
    assert rc == -1 and b"go together" in lib.asis_last_error()
    rc = lib.asis_frames_to_batch(None, fake, None, None, 2, 8, 8, None)
    assert rc == -1 and b"null pointer" in lib.asis_last_error()


def test_host_side_validation_last_build_entry_points():
    """Host logic touched by the last build of round 2: the depth-wise convolution stages its taps in shared memory
    (channel limit reported, not silently exceeded), its backward workspace follows the one-wave grid, and the
    LayerNorm backward workspace follows the 4-blocks-per-SM grid."""
    import ctypes
    from adaptersis_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(256)
    hs = (ctypes.c_int * 2)(7, 4)
    ws = (ctypes.c_int * 2)(5, 3)
    rc = lib.asis_dwconv3x3_forward(fake, 1, fake, fake, None, fake, 2, 1284, 2, hs, ws, 1, None)
    assert rc == -1 and b"1280" in lib.asis_last_error()
    rc = lib.asis_dwconv3x3_forward(fake, 1, fake, fake, None, fake, 2, 66, 2, hs, ws, 1, None)
    assert rc == -1 and b"multiple of 4" in lib.asis_last_error()
    rc = lib.asis_dwconv3x3_forward(fake, 1, fake, fake, None, fake, 2, 64, 0, hs, ws, 1, None)
    assert rc == -1 and b"maps required" in lib.asis_last_error()
    # backward: partials of at most 296 blocks over all channel blocks (one wave of two blocks per SM) + the GELU' buffer
    for C, ntok in ((256, 6949), (64, 47), (1024, 6949)):
        need = lib.asis_dwconv3x3_backward_workspace_bytes(12, C, ntok)
        rows = 12 * ntok
        rb = min((rows + 63) // 64, max(1, 296 // ((C + 127) // 128)))
        assert need == (rb * 10 * C * 4 + 255) // 256 * 256 + 12 * ntok * C * 4, (C, ntok, need)
    rc = lib.asis_dwconv3x3_backward(fake, fake, fake, 1, fake, fake, fake, fake, 0, 12, 256, 2, hs, ws, 1, fake, 16, None)
    assert rc != 0 and b"workspace" in lib.asis_last_error()
    # LayerNorm backward: 2 rows per block iteration, at most 4 x 148 persistent blocks, two partial rows of C floats per block
    assert lib.asis_layernorm_backward_workspace_bytes(21168, 1024) == 592 * 2 * 1024 * 4
    assert lib.asis_layernorm_backward_workspace_bytes(100, 1024) == 50 * 2 * 1024 * 4
    rc = lib.asis_layernorm_backward(fake, 1, fake, 0, fake, fake, fake, None, fake, None, None, 0, 64, 1024, fake, 16, None)
    assert rc != 0 and b"workspace" in lib.asis_last_error()
    rc = lib.asis_layernorm_backward(fake, 1, fake, 0, fake, fake, fake, None, fake, None, None, 0, 64, 2048, fake, 1 << 20, None)
    assert rc != 0 and b"1024" in lib.asis_last_error()


def test_dwconv_backward_refuses_misaligned_pointers():
    """The depth-wise convolution backward loads and stores 4-channel vectors of dy, pre, x and dx (and of the GELU'
    buffer in the workspace): a pointer off the 16-byte grid is refused on the host, before any launch."""
    import ctypes
    from adaptersis_b200 import _lib
    lib = _lib.load()
    fake, odd = ctypes.c_void_p(256), ctypes.c_void_p(260)
    hs = (ctypes.c_int * 2)(7, 4)
    ws = (ctypes.c_int * 2)(5, 3)
    need = lib.asis_dwconv3x3_backward_workspace_bytes(2, 64, 47)
    for dtype in (0, 1):
        for i in range(5):                       # dy, pre, x, dx, workspace
            p = [fake] * 5
            p[i] = odd
            rc = lib.asis_dwconv3x3_backward(p[0], p[1], p[2], dtype, fake, p[3], fake, fake, 0, 2, 64, 2, hs, ws, 1,
                                             p[4], need, None)
            assert rc == -1 and b"16-byte aligned" in lib.asis_last_error(), i


def test_no_cpu_fallback():
    import adaptersis_b200 as asis
    m = asis.MSDeformAttn(d_model=32, n_levels=1, n_heads=4, n_points=2)
    q = torch.randn(1, 4, 32)
    ref = torch.rand(1, 4, 1, 2)
    ss = torch.tensor([[2, 2]])
    with pytest.raises(RuntimeError, match="CUDA"):
        m(q, ref, q, ss, torch.tensor([0]))
    blk = asis.Block(dim=32, num_heads=2, init_values=1e-5)
    with pytest.raises(RuntimeError, match="CUDA"):
        blk(torch.randn(1, 3, 32))


def test_missing_library_fails_loudly(monkeypatch):
    from adaptersis_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libasis_b200.so")
    with pytest.raises(RuntimeError, match="no CPU or library fallback"):
        _lib.load()
