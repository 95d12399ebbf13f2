"""Multi-scale deformable attention kernels against fp64 with elementwise bounds (tests/msda_ref.py), in every template
instantiation the launcher can pick, in both value dtypes, with samples on cell borders, on and just inside the map's
edges and far outside.  Every case asserts from the torch.profiler trace which instantiation ran with which grid (the
launcher's arithmetic below), prints the launches and the worst err / bound ratio with where it occurred, and the
backward is run twice and must be bit-identical.  The sweep calls the C ABI with each output inside a NaN-filled
buffer: nothing outside the outputs may change."""
import time

import pytest
import torch

import msda_ref as MR
import tc_ref as R
from adaptersis_b200 import _lib, kernels as K
from adaptersis_b200._lib import ptr
from tc_ref import bits, guarded, guards_intact

pytestmark = pytest.mark.gpu
DEV = "cuda"
BF, F32 = torch.bfloat16, torch.float32
VT = {F32: "float", BF: "__nv_bfloat16"}


# ------------------------------------------------------------------------------- the launcher's arithmetic
def _ipb(gp, LP, entry_bytes):
    ipb = 256 // gp
    while ipb * gp > 32 and ipb * LP * entry_bytes > 40 * 1024:
        ipb >>= 1
    return ipb


def launch_plan(dtype, N, S, M, D, Lq, L, P):
    """{kernel: (instantiation, grid)} of one forward and one backward, as launch_fwd / launch_bwd choose them."""
    cpl = 8 if dtype == BF and D % 8 == 0 else 4
    gp = max(4, MR.group_pad(D // cpl))
    ipb = _ipb(gp, L * P, 32)
    lgp = MR.locaw_gp(D)
    lipb = _ipb(lgp, L * P, 48)
    kc = (Lq + 255) // 256
    cap = max(1, (256 << 20) // (N * M * S * 4))
    kc = min(kc, cap)
    qchunk = -(-Lq // kc)
    KC = -(-Lq // qchunk)
    full = "true" if D == 16 * lgp else "false"
    return {
        "fwd": (f"msda_fwd_kernel<{VT[dtype]},{cpl},{gp}>", (-(-Lq // ipb), M, N)),
        "locaw": (f"msda_bwd_locaw_kernel<{VT[dtype]},{cpl},{lgp},{full}>", (-(-Lq // lipb), M, N)),
        "scan": ("msda_bwd_scan_kernel", (N * M,)),
        "fill": (f"msda_bwd_fill_kernel<{'true' if qchunk * P <= 65535 else 'false'}>", (KC, L, N * M)),
        "gather": (f"msda_bwd_gather_kernel<{VT[dtype]},{cpl},{gp}>", (-(-S // (256 // gp)), M, N)),
    }


def reachable():
    """Every instantiation of the forward, locaw, gather and fill kernels some valid (dtype, D) reaches."""
    names = {"msda_bwd_fill_kernel<true>", "msda_bwd_fill_kernel<false>"}
    for dtype in (F32, BF):
        for D in range(4, 129, 4):
            plan = launch_plan(dtype, 1, 64, 1, D, 64, 1, 4)
            names |= {plan[k][0] for k in ("fwd", "locaw", "gather")}
    return names


def expect_launches(ks, plan, kinds):
    """The trace holds exactly one launch of each kernel of `kinds`, with the planned instantiation and grid."""
    assert len([k for k in ks if "msda_" in k[0]]) == len(kinds), ks
    for kind in kinds:
        R.expect_kernel(ks, "asis::" + plan[kind][0] + "(", plan[kind][1])


# ------------------------------------------------------------------------------------------------ helpers
def lsi_of(ss):
    return torch.cat([ss.new_zeros(1), ss.prod(1).cumsum(0)[:-1]])


def report(tag, reps, plan, t0):
    worst = max(reps, key=lambda r: r.ratio)
    print(f"[{tag}] {plan['fwd'][0]} {plan['locaw'][0]} {plan['fill'][0]} {plan['gather'][0]}; "
          f"max err/bound {worst.ratio:.3g} ({worst.name} at {worst.where}) [{time.time() - t0:.1f} s]")
    for r in reps:
        assert r.ok, f"[{tag}] {r}"


def abi_forward(value, ss, lsi, loc, aw):
    N, S, M, D = value.shape
    _, Lq, _, L, P, _ = loc.shape
    buf, out = guarded((N, Lq, M * D), value.dtype)
    _lib.check(_lib.load().asis_msda_forward(ptr(value), _lib.dt(value), ptr(ss), ptr(lsi), ptr(loc), ptr(aw),
                                             ptr(out), _lib.dt(out), N, S, M, D, Lq, L, P, _lib.stream()))
    return out, [buf]


def abi_backward(value, ss, lsi, loc, aw, gout):
    N, S, M, D = value.shape
    _, Lq, _, L, P, _ = loc.shape
    lib = _lib.load()
    bv, gv = guarded(tuple(value.shape), value.dtype)
    bl, gl = guarded(tuple(loc.shape), F32)
    ba, ga = guarded(tuple(aw.shape), F32)
    nbytes = lib.asis_msda_backward_workspace_bytes(N, S, M, D, Lq, L, P)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    _lib.check(lib.asis_msda_backward(ptr(value), _lib.dt(value), ptr(ss), ptr(lsi), ptr(loc), ptr(aw), ptr(gout),
                                      _lib.dt(gout), ptr(gv), ptr(gl), ptr(ga), N, S, M, D, Lq, L, P, ptr(ws), nbytes,
                                      _lib.stream()))
    return (gv, gl, ga), [bv, bl, ba]


def run_case(tag, value, shapes, loc, aw, gout, abi=False):
    """Forward and backward (traced, planned launches asserted), the bounds, the backward's run-to-run identity."""
    t0 = time.time()
    N, S, M, D = value.shape
    _, Lq, _, L, P, _ = loc.shape
    ss = torch.as_tensor(shapes, dtype=torch.long, device=DEV)
    lsi = lsi_of(ss)
    value, loc, aw, gout = value.to(DEV), loc.to(DEV).float(), aw.to(DEV).float(), gout.to(DEV).to(value.dtype)
    plan = launch_plan(value.dtype, N, S, M, D, Lq, L, P)
    inputs = [t.clone() for t in (value, loc, aw, gout)]
    if abi:
        (out, bufs), ks = R.traced(lambda: abi_forward(value, ss, lsi, loc, aw))
        ((gv, gl, ga), bufs_b), kb = R.traced(lambda: abi_backward(value, ss, lsi, loc, aw, gout))
        assert all(guards_intact(b) for b in bufs + bufs_b), f"[{tag}] a kernel wrote outside its output"
        assert all(torch.equal(bits(a), bits(b)) for a, b in zip(inputs, (value, loc, aw, gout))), "input modified"
        again, _ = abi_backward(value, ss, lsi, loc, aw, gout)
    else:
        out, ks = R.traced(lambda: K.msda_forward(value, ss, lsi, loc, aw))
        (gv, gl, ga), kb = R.traced(lambda: K.msda_backward(value, ss, lsi, loc, aw, gout))
        again = K.msda_backward(value, ss, lsi, loc, aw, gout)
    expect_launches(ks, plan, ["fwd"])
    expect_launches(kb, plan, ["locaw", "scan", "fill", "gather"])
    for a, b in zip((gv, gl, ga), again):
        assert torch.equal(bits(a), bits(b)), f"[{tag}] the backward is not run-to-run identical"
    refs = MR.msda_refs(value, shapes, loc, aw, gout)
    reps = MR.check_all(dict(out=out, grad_value=gv, grad_loc=gl, grad_attn=ga), refs, value.dtype, shapes)
    del refs
    report(tag, reps, plan, t0)


# ------------------------------------------------------------------------------------- instantiation sweep
SWEEP_SHAPES = [(13, 21), (7, 5), (1, 3)]
SWEEP = [(F32, D) for D in (8, 16, 24, 32, 48, 64, 96, 128)] + \
        [(BF, D) for D in (8, 16, 24, 32, 48, 64, 96, 128, 12, 20, 36, 100)]


def sweep_inputs(dtype, D, seed):
    g = torch.Generator().manual_seed(seed)
    N, M, P, Lq = 2, 3, 4, 777
    value, gout = MR.operands(g, N, Lq, M, D, SWEEP_SHAPES, dtype)
    loc = MR.sample_locations(g, N, Lq, M, SWEEP_SHAPES, P)
    aw = MR.attention_weights(g, N, Lq, M, len(SWEEP_SHAPES), P)
    return value, loc, aw, gout


@pytest.mark.parametrize("dtype,D", SWEEP, ids=[f"{'bf16' if d == BF else 'f32'}-D{D}" for d, D in SWEEP])
def test_sweep(dtype, D):
    value, loc, aw, gout = sweep_inputs(dtype, D, 100 + D)
    run_case(f"sweep {dtype} D={D}", value, SWEEP_SHAPES, loc, aw, gout, abi=True)


SPARSE_SHAPES = [(40, 50), (7, 5), (1, 3)]


@pytest.mark.parametrize("dtype", [F32, BF])
def test_untouched_pixels_exactly_zero(dtype):
    """grad_value is exactly 0 (not merely small) at the pixels that no in-map corner touches: a 40 x 50 level that
    the samples of 100 queries cannot cover."""
    g = torch.Generator().manual_seed(7)
    N, M, D, P, Lq = 2, 3, 64, 4, 100
    value, gout = MR.operands(g, N, Lq, M, D, SPARSE_SHAPES, dtype)
    loc = MR.sample_locations(g, N, Lq, M, SPARSE_SHAPES, P)
    aw = MR.attention_weights(g, N, Lq, M, len(SPARSE_SHAPES), P)
    ss = torch.as_tensor(SPARSE_SHAPES, dtype=torch.long, device=DEV)
    ld = loc.to(DEV)
    gv, _, _ = K.msda_backward(value.to(DEV), ss, lsi_of(ss), ld, aw.to(DEV), gout.to(DEV))
    geo = MR.geometry(ld, SPARSE_SHAPES)
    S = value.shape[1]
    touched = torch.zeros(N, S, M, dtype=torch.bool, device=DEV)
    nn = torch.arange(N, device=DEV).view(N, 1, 1, 1, 1, 1).expand_as(geo["pix"])
    mm = torch.arange(M, device=DEV).view(1, 1, M, 1, 1, 1).expand_as(geo["pix"])
    touched[nn[geo["mask"]], geo["pix"][geo["mask"]], mm[geo["mask"]]] = True
    assert (~touched).sum() > 0 and touched.sum() > 0
    assert bool((gv[~touched] == 0).all())
    assert bool((gv[touched].float().abs().amax(-1) > 0).any())


# -------------------------------------------------------------------------------------- production shapes
def module_locations(N, Lq, M, shapes, ref, dtype, seed):
    """Sampling locations and attention weights from the prep kernel applied to MSDeformAttn's bias-grid offsets
    (plus a spread of 0.5 px per point) and to the given reference points."""
    from adaptersis_b200.ms_deform_attn import MSDeformAttn
    L, P = len(shapes), 4
    g = torch.Generator().manual_seed(seed)
    bias = MSDeformAttn(d_model=M * 8, n_levels=L, n_heads=M, n_points=P).sampling_offsets.bias.detach()
    off = bias + 0.5 * torch.randn(N, Lq, M * L * P * 2, generator=g)
    logits = torch.randn(N, Lq, M * L * P, generator=g)
    ss = torch.as_tensor(shapes, dtype=torch.long, device=DEV)
    return K.msda_prep_forward(off.to(DEV).to(dtype), logits.to(DEV).to(dtype), ref, ss, N, Lq, M, L, P)


def deform_refs():
    from adaptersis_b200 import deform_inputs
    d1, d2 = deform_inputs(torch.empty(1, 3, 588, 588, device=DEV), 14)
    return d1[0], d2[0]


PRODUCTION = [(dtype, N, M, D, which) for dtype in (F32, BF) for (M, D) in ((8, 128), (12, 64))
              for which in ("injector", "extractor") for N in (2,)] + [(BF, 12, 8, 128, "injector")]


@pytest.mark.parametrize("dtype,N,M,D,which", PRODUCTION,
                         ids=[f"{w}-{'bf16' if d == BF else 'f32'}-N{n}-M{m}-D{dd}" for d, n, m, dd, w in PRODUCTION])
def test_production_shapes(dtype, N, M, D, which):
    inj, ext = deform_refs()
    if which == "injector":
        shapes, Lq, ref = [(73, 73), (36, 36), (18, 18)], 1764, inj
    else:
        shapes, Lq, ref = [(42, 42)], 6949, ext
    assert ref.shape[1] == Lq
    loc, aw = module_locations(N, Lq, M, shapes, ref, dtype, seed=N + M)
    g = torch.Generator().manual_seed(D + M)
    value, gout = MR.operands(g, N, Lq, M, D, shapes, dtype)
    run_case(f"{which} {dtype} N={N} M={M} D={D}", value, shapes, loc, aw, gout)


# ---------------------------------------------------------------------------------------------- limits
LIMIT_SHAPES = [(9, 11), (1, 7), (5, 1), (3, 3), (6, 2), (2, 6), (1, 1), (4, 5)]


@pytest.mark.parametrize("dtype,D", [(F32, 8), (F32, 128), (BF, 8), (BF, 128)])
def test_eight_levels_eight_points(dtype, D):
    """L P = 64: at D <= 16 the locaw block shrinks to one warp with 96 KB of shared memory."""
    g = torch.Generator().manual_seed(D)
    N, M, P, Lq = 2, 2, 8, 301
    value, gout = MR.operands(g, N, Lq, M, D, LIMIT_SHAPES, dtype)
    loc = MR.sample_locations(g, N, Lq, M, LIMIT_SHAPES, P)
    aw = MR.attention_weights(g, N, Lq, M, len(LIMIT_SHAPES), P)
    run_case(f"L8 P8 {dtype} D={D}", value, LIMIT_SHAPES, loc, aw, gout, abi=True)


@pytest.mark.parametrize("name,N,Lq,M,D,shapes,P", [
    ("fill_windows", 1, 3000, 2, 8, [(300, 300)], 4),          # a level over 81920 pixels: cursor windows
    ("fill_int_cursors", 12, 17000, 16, 8, [(424, 424)], 4),   # qchunk * P > 65535: 32-bit cursors
])
def test_bf16_large_value_maps(name, N, Lq, M, D, shapes, P):
    g = torch.Generator().manual_seed(21)
    value, gout = MR.operands(g, N, Lq, M, D, shapes, BF)
    loc = torch.rand(N, Lq, M, len(shapes), P, 2, generator=g) * 1.04 - 0.02
    loc[:, ::2] = loc[:, ::2] * 0.05                            # half of the samples in one corner: long lists
    aw = MR.attention_weights(g, N, Lq, M, len(shapes), P)
    run_case(f"{name} bf16", value, shapes, loc, aw, gout)


LARGE = {"fill_windows": (BF, 1, 90000, 2, 8, 3000, 1, 4), "fill_int_cursors": (BF, 12, 179776, 16, 8, 17000, 1, 4)}


# --------------------------------------------------------------------------------------------------- prep
PREP_SHAPES = [(13, 21), (7, 5), (1, 3)]


@pytest.mark.parametrize("dtype", [F32, BF])
@pytest.mark.parametrize("ref_dim", [2, 4])
@pytest.mark.parametrize("rows", ["Lq", "NLq"])
@pytest.mark.parametrize("levels", [1, 3])
def test_prep(dtype, ref_dim, rows, levels):
    N, Lq, M, P = 2, 333, 3, 4
    L = len(PREP_SHAPES)
    g = torch.Generator().manual_seed(ref_dim + 10 * levels)
    off = (torch.randn(N, Lq, M * L * P * 2, generator=g) * 3).to(dtype).to(DEV)
    logits = (torch.randn(N, Lq, M * L * P, generator=g) * 4).to(dtype)
    logits[:, ::9] *= 8                                         # rows with a wide range: tiny weights
    logits = logits.to(DEV)
    ref = torch.rand(N if rows == "NLq" else 1, Lq, levels, ref_dim, generator=g)
    if ref_dim == 4:
        ref[..., 2:] = ref[..., 2:] * 0.5 + 0.05
    ref = ref.to(DEV)
    ss = torch.as_tensor(PREP_SHAPES, dtype=torch.long, device=DEV)
    loc, attn = K.msda_prep_forward(off, logits, ref, ss, N, Lq, M, L, P)
    rf = MR.prep_forward_refs(off, logits, ref, PREP_SHAPES, N, Lq, M, L, P)
    gloc = torch.randn(N, Lq, M, L, P, 2, generator=g).to(DEV)
    gattn = torch.randn(N, Lq, M, L, P, generator=g).to(DEV)
    goff, glog = K.msda_prep_backward(gloc, gattn, attn, ref, ss, dtype, N, Lq, M, L, P)
    rb = MR.prep_backward_refs(gloc, gattn, attn, ref, PREP_SHAPES, dtype, N, Lq, M, L, P)
    reps = [R.check(k, o.reshape(rf[k][0].shape), rf[k][0], R.U_F32, rf[k][1], block=MR.query_slabs)
            for k, o in (("loc", loc), ("attn", attn))]
    reps += [R.check(k, o.reshape(rb[k][0].shape), rb[k][0], R.u_out(dtype), rb[k][1], block=MR.query_slabs)
             for k, o in (("grad_offsets", goff), ("grad_logits", glog))]
    worst = max(reps, key=lambda r: r.ratio)
    print(f"[prep {dtype} ref_dim={ref_dim} rows={rows} levels={levels}] max err/bound {worst.ratio:.3g} "
          f"({worst.name} at {worst.where})")
    for r in reps:
        assert r.ok, str(r)


# ------------------------------------------------------------------------------------------------ coverage
def test_every_instantiation_asserted():
    """The cases above assert, together, every reachable instantiation of the forward, locaw, gather and fill
    kernels (each case asserts its launch_plan, so the union of the plans is what the file asserts)."""
    asserted = set()
    for dtype, D in SWEEP:
        plan = launch_plan(dtype, 2, sum(h * w for h, w in SWEEP_SHAPES), 3, D, 777, len(SWEEP_SHAPES), 4)
        asserted |= {plan[k][0] for k in ("fwd", "locaw", "fill", "gather")}
    for args in LARGE.values():
        asserted.add(launch_plan(*args)["fill"][0])
    missing = reachable() - asserted
    assert not missing, f"instantiations no case asserts: {sorted(missing)}"
    print(f"[coverage] {len(asserted)} instantiations asserted; peak memory "
          f"{torch.cuda.max_memory_allocated() / 2 ** 30:.2f} GB")
