"""GPU parity tests of the MSDA operator through the C-ABI (visionllm_b200.msda),
against the CPU oracle (oracle/msda_oracle.c) and the reference-generated golden
vectors.  Mirrors mmcv/tests/test_ops/test_ms_deformable_attn.py."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import msda_oracle as O  # noqa: E402


def _ext():
    import visionllm_b200.msda as ext
    return ext


def _dev(*arrs, dtype=None):
    out = []
    for a in arrs:
        t = torch.from_numpy(np.ascontiguousarray(a))
        if dtype is not None and t.is_floating_point():
            t = t.to(dtype)
        out.append(t.cuda())
    return out


def make_case(shapes_l, N, M, D, Lq, P, seed, lo=-0.15, hi=1.15):
    rng = np.random.default_rng(seed)
    shapes = np.array(shapes_l, dtype=np.int64)
    L = len(shapes_l)
    S = int(shapes.prod(1).sum())
    lsi = np.concatenate([[0], np.cumsum(shapes.prod(1))[:-1]]).astype(np.int64)
    value = rng.standard_normal((N, S, M, D), dtype=np.float32)
    loc = (rng.random((N, Lq, M, L, P, 2), dtype=np.float32) * (hi - lo) + lo).astype(np.float32)
    attw = rng.random((N, Lq, M, L, P), dtype=np.float32) + 1e-3
    attw = (attw / attw.sum((-1, -2), keepdims=True)).astype(np.float32)
    return value, shapes, lsi, loc, attw


# ---- the mmcv unit-test vector ---------------------------------------------------
def test_mmcv_seed3_fp64(golden_dir):
    g = np.load(os.path.join(golden_dir, "msda_mmcv_seed3.npz"))
    v, sh, lsi, loc, w = _dev(g["value"].astype(np.float64), g["shapes"], g["lsi"], g["loc"].astype(np.float64),
                              g["attw"].astype(np.float64))
    out = _ext().ms_deform_attn_forward(v, sh, lsi, loc, w, 2).cpu().numpy().reshape(g["out_f64"].shape)
    ref = g["out_f64"]
    assert np.abs(out - ref).max() < 1e-18           # test_ms_deformable_attn.py:99-102
    assert (np.abs(out - ref) / np.abs(ref)).max() < 1e-15


@pytest.mark.parametrize("flags", [0, 1])
def test_mmcv_seed3_fp32(golden_dir, flags):
    g = np.load(os.path.join(golden_dir, "msda_mmcv_seed3.npz"))
    v, sh, lsi, loc, w = _dev(g["value"], g["shapes"], g["lsi"], g["loc"], g["attw"])
    out = _ext().ms_deform_attn_forward(v, sh, lsi, loc, w, 2, flags=flags).cpu().numpy()
    ref = g["out_f32"].reshape(out.shape)
    assert np.allclose(out, ref, rtol=1e-2, atol=1e-3)   # :129
    assert np.abs(out - ref).max() < 1e-9                 # :133
    assert (np.abs(out - ref) / np.abs(ref)).max() < 1e-6  # :134


# ---- strict kernel: bit-exact against the C oracle ---------------------------------
CASES = [
    ([(13, 17), (7, 9), (4, 5), (2, 3)], 2, 8, 32, 37, 4),
    ([(100, 37)], 1, 2, 32, 64, 4),
    ([(9, 11), (5, 6)], 3, 3, 16, 21, 2),
    ([(8, 7)], 1, 2, 71, 9, 5),
    ([(6, 4), (3, 2), (2, 2), (1, 1), (1, 1)], 2, 4, 32, 11, 4),   # K = 20
    ([(5, 5), (3, 3), (2, 2)], 1, 8, 32, 130, 4),                  # K = 12
    ([(30, 40)], 2, 8, 32, 50, 32),                                # K = 32
    ([(30, 40)], 1, 2, 32, 7, 40),                                 # K = 40 -> strict path
    ([(3, 3)], 1, 1, 4, 1, 1),
]


@pytest.mark.parametrize("case", CASES, ids=[str(i) for i in range(len(CASES))])
def test_strict_fp32_bit_exact_vs_oracle(case):
    value, shapes, lsi, loc, attw = make_case(*case, seed=100 + len(case[0]))
    ref = O.forward_kernel_semantics(value, shapes, lsi, loc, attw)
    v, sh, ls, lo, w = _dev(value, shapes, lsi, loc, attw)
    out = _ext().ms_deform_attn_forward(v, sh, ls, lo, w, 64, flags=1).cpu().numpy()
    assert out.dtype == np.float32 and out.shape == ref.shape
    assert np.array_equal(out.view(np.uint32), ref.view(np.uint32)), np.abs(out - ref).max()


@pytest.mark.parametrize("case", CASES[:3], ids=["0", "1", "2"])
def test_strict_fp64_bit_exact_vs_oracle(case):
    value, shapes, lsi, loc, attw = make_case(*case, seed=7)
    value, loc, attw = value.astype(np.float64), loc.astype(np.float64), attw.astype(np.float64)
    ref = O.forward_kernel_semantics(value, shapes, lsi, loc, attw)
    v, sh, ls, lo, w = _dev(value, shapes, lsi, loc, attw)
    out = _ext().ms_deform_attn_forward(v, sh, ls, lo, w, 64).cpu().numpy()
    assert np.array_equal(out.view(np.uint64), ref.view(np.uint64))


# ---- fast kernel: indices bit-exact, values within fp32 reassociation noise ---------
@pytest.mark.parametrize("variant", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("case", [c for c in CASES if c[3] == 32 and len(c[0]) * c[5] <= 32],
                         ids=lambda c: f"L{len(c[0])}P{c[5]}Lq{c[4]}")
def test_fast_fp32_vs_oracle(case, variant):
    ext = _ext()
    from visionllm_b200 import _lib
    value, shapes, lsi, loc, attw = make_case(*case, seed=5)
    ref = O.forward_kernel_semantics(value, shapes, lsi, loc, attw)
    v, sh, ls, lo, w = _dev(value, shapes, lsi, loc, attw)
    _lib.lib().vllm_msda_set_variant(variant)
    try:
        out = ext.ms_deform_attn_forward(v, sh, ls, lo, w, 64).cpu().numpy()
    finally:
        _lib.lib().vllm_msda_set_variant(0)
    # north-star tolerance is 1e-3 rel; reassociation of <= 4*K fp32 terms gives ~1e-6
    assert np.abs(out - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max())


@pytest.mark.parametrize("shapes_l", [[(13, 17), (100, 37)], [(128, 128), (64, 64), (32, 32), (16, 16)]])
def test_sampling_indices_bit_exact(shapes_l):
    rng = np.random.default_rng(3)
    shapes = np.array(shapes_l, dtype=np.int64)
    L = len(shapes_l)
    loc = (rng.random((2, 500, 8, L, 4, 2), dtype=np.float32) * 1.3 - 0.15).astype(np.float32)
    # adversarial: pixel centres of each level, replicated over the level axis (SURVEY Appendix A)
    for l, (H, W) in enumerate(shapes_l):
        n = min(500, W)
        loc[0, :n, 0, :, 0, 0] = ((np.arange(n, dtype=np.float32) + np.float32(0.5)) / np.float32(W))[:, None]
        n = min(500, H)
        loc[0, :n, 0, :, 0, 1] = ((np.arange(n, dtype=np.float32) + np.float32(0.5)) / np.float32(H))[:, None]
    ref = O.sample_indices(shapes, loc)
    sh, lo = _dev(shapes, loc)
    got = _ext().ms_deform_attn_sample_indices(sh, lo).cpu().numpy()
    assert np.array_equal(got, ref)
    assert (got[..., 2] & 1).any() and ((got[..., 2] & 1) == 0).any()


# ---- reference-generated golden vectors ----------------------------------------------
@pytest.mark.parametrize("name", ["msda_ref_d32_npot.npz", "msda_ref_d32_pixel.npz", "msda_ref_d16_l2p2.npz",
                                  "msda_ref_d71_l1p5.npz"])
@pytest.mark.parametrize("flags", [0, 1])
def test_golden_reference_outputs(golden_dir, name, flags):
    g = np.load(os.path.join(golden_dir, name))
    v, sh, lsi, loc, w = _dev(g["value"], g["shapes"], g["lsi"], g["loc"], g["attw"])
    out = _ext().ms_deform_attn_forward(v, sh, lsi, loc, w, 64, flags=flags).cpu().numpy()
    ref = g["out_f64"].reshape(out.shape)
    # fp32 kernel vs the reference's fp64 grid_sample output: <= 1e-3 rel is the north-star bound
    assert np.abs(out - ref).max() <= 2e-5 * max(1.0, np.abs(ref).max())


# ---- edge cases and error behaviour ---------------------------------------------------
def test_empty_inputs():
    ext = _ext()
    value, shapes, lsi, loc, attw = make_case([(4, 4)], 2, 8, 32, 5, 4, seed=1)
    v, sh, ls, lo, w = _dev(value, shapes, lsi, loc, attw)
    out = ext.ms_deform_attn_forward(v, sh, ls, lo[:, :0].contiguous(), w[:, :0].contiguous(), 64)
    assert out.shape == (2, 0, 256)


def test_all_samples_out_of_range_gives_zeros():
    value, shapes, lsi, loc, attw = make_case([(4, 4), (2, 2)], 1, 8, 32, 9, 4, seed=1, lo=1.5, hi=3.0)
    v, sh, ls, lo, w = _dev(value, shapes, lsi, loc, attw)
    for flags in (0, 1):
        out = _ext().ms_deform_attn_forward(v, sh, ls, lo, w, 64, flags=flags)
        assert torch.count_nonzero(out).item() == 0


def test_nan_in_unsampled_value_does_not_leak():
    value, shapes, lsi, loc, attw = make_case([(8, 8)], 1, 8, 32, 16, 4, seed=2, lo=0.3, hi=0.6)
    value[0, :8] = np.nan      # first row is never touched by samples in [0.3, 0.6]
    value[0, -8:] = np.inf
    v, sh, ls, lo, w = _dev(value, shapes, lsi, loc, attw)
    for flags in (0, 1):
        out = _ext().ms_deform_attn_forward(v, sh, ls, lo, w, 64, flags=flags)
        assert torch.isfinite(out).all()


def test_error_behaviour_matches_reference():
    ext = _ext()
    value, shapes, lsi, loc, attw = make_case([(4, 4)], 3, 2, 32, 5, 4, seed=1)
    v, sh, ls, lo, w = _dev(value, shapes, lsi, loc, attw)
    with pytest.raises(RuntimeError):       # non-contiguous (ms_deform_attn_cuda.cu:215-224)
        ext.ms_deform_attn_forward(v.transpose(1, 2), sh, ls, lo, w, 64)
    with pytest.raises(RuntimeError):       # CPU tensor (:226-231)
        ext.ms_deform_attn_forward(v.cpu(), sh, ls, lo, w, 64)
    with pytest.raises(RuntimeError):       # batch % im2col_step (:244-245)
        ext.ms_deform_attn_forward(v, sh, ls, lo, w, 2)
    with pytest.raises(RuntimeError):       # half is not dispatched (AT_DISPATCH_FLOATING_TYPES, :258)
        ext.ms_deform_attn_forward(v.half(), sh, ls, lo.half(), w.half(), 64)
    ext.ms_deform_attn_forward(v, sh, ls, lo, w, 3)
    ext.ms_deform_attn_forward(v, sh, ls, lo, w, im2col_step=1)   # mmcv keyword flavour


# ---- BASELINE full size: size-independent properties ------------------------------------
def _full_size(N=8, Lq=None, seed=0):
    shapes_l = [(128, 128), (64, 64), (32, 32), (16, 16)]
    g = torch.Generator(device="cuda").manual_seed(seed)
    shapes = torch.tensor(shapes_l, dtype=torch.int64, device="cuda")
    lsi = torch.cat((shapes.new_zeros(1), shapes.prod(1).cumsum(0)[:-1]))
    S = int(shapes.prod(1).sum())
    Lq = S if Lq is None else Lq
    value = torch.randn(N, S, 8, 32, device="cuda", generator=g)
    loc = torch.rand(N, Lq, 8, 4, 4, 2, device="cuda", generator=g) * 1.1 - 0.05
    attw = torch.softmax(torch.randn(N, Lq, 8, 16, device="cuda", generator=g), -1).view(N, Lq, 8, 4, 4)
    return value, shapes, lsi, loc, attw


def test_full_size_fast_equals_strict_and_hint_invariance():
    ext = _ext()
    value, shapes, lsi, loc, attw = _full_size()
    fast = ext.ms_deform_attn_forward(value, shapes, lsi, loc, attw, 64)
    strict = ext.ms_deform_attn_forward(value, shapes, lsi, loc, attw, 64, flags=1)
    assert (fast - strict).abs().max().item() <= 1e-5 * strict.abs().max().item()
    # the host shape hint only re-orders work: results must be bit-identical without it
    from visionllm_b200 import _lib
    _lib.lib().vllm_msda_set_variant(4)
    try:
        nohint = ext.ms_deform_attn_forward(value, shapes, lsi, loc, attw, 64)
    finally:
        _lib.lib().vllm_msda_set_variant(0)
    assert torch.equal(fast, nohint)


def test_full_size_constant_value_partition_of_unity():
    ext = _ext()
    value, shapes, lsi, loc, attw = _full_size(N=2)
    value.fill_(1.0)
    loc = loc.clamp(0.2, 0.8)      # strictly interior: every bilinear stencil sums to 1
    out = ext.ms_deform_attn_forward(value, shapes, lsi, loc.contiguous(), attw, 64)
    assert (out - 1.0).abs().max().item() < 1e-5


def test_full_size_linearity_in_value():
    ext = _ext()
    value, shapes, lsi, loc, attw = _full_size(N=2, Lq=900)
    v2 = torch.randn_like(value)
    a = ext.ms_deform_attn_forward(value, shapes, lsi, loc, attw, 64)
    b = ext.ms_deform_attn_forward(v2, shapes, lsi, loc, attw, 64)
    c = ext.ms_deform_attn_forward(value * 2 + v2, shapes, lsi, loc, attw, 64)
    assert (c - (2 * a + b)).abs().max().item() < 1e-4


# ---- "fast mode" (SURVEY 8d cfg 2b): bf16 value read in place ----
@pytest.mark.parametrize("case", ["enc", "dec", "oob", "odd_points"])
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.bfloat16])
def test_bf16_value_matches_fp32_op_on_upcast_value(case, out_dtype):
    """ms_deform_attn_forward_bf16(value_bf16) == ms_deform_attn_forward(value_bf16.float()) (exact upcast inside the
    kernel, same fp32 FMAs up to summation order) and vs the C oracle on the upcast value."""
    import visionllm_b200.msda as ext
    from oracle import msda_oracle as O
    g = torch.Generator(device="cuda").manual_seed(7)
    shapes_l = [(20, 27), (10, 14), (5, 7), (3, 4)]
    L, P = (4, 4) if case != "odd_points" else (4, 3)
    shapes = torch.tensor(shapes_l, dtype=torch.int64, device="cuda")
    lsi = torch.cat((shapes.new_zeros(1), shapes.prod(1).cumsum(0)[:-1]))
    S = int(shapes.prod(1).sum())
    N, M, D = 3, 8, 32
    Lq = S if case != "dec" else 37
    value = torch.randn(N, S, M, D, device="cuda", generator=g).bfloat16()
    spread = 1.6 if case == "oob" else 1.0
    loc = (torch.rand(N, Lq, M, L, P, 2, device="cuda", generator=g) - 0.5) * spread + 0.5
    aw = torch.softmax(torch.randn(N, Lq, M, L * P, device="cuda", generator=g), -1).view(N, Lq, M, L, P).contiguous()
    fast = ext.ms_deform_attn_forward_bf16(value, shapes, lsi, loc, aw, out_dtype)
    ref = ext.ms_deform_attn_forward(value.float(), shapes, lsi, loc, aw, 64)
    orc = torch.from_numpy(O.forward_kernel_semantics(value.float().cpu().numpy(), shapes.cpu().numpy(), lsi.cpu().numpy(),
                                                      loc.cpu().numpy(), aw.cpu().numpy())).cuda()
    assert fast.dtype == out_dtype and fast.shape == ref.shape
    scale = orc.abs().max().item()
    if out_dtype == torch.float32:
        assert (fast - ref).abs().max().item() <= 1e-5 * scale
        assert (fast - orc).abs().max().item() <= 1e-5 * scale
    else:
        assert torch.equal(fast, ref.bfloat16()) or ((fast.float() - ref).abs() <= 2.0 ** -8 * ref.abs() + 1e-5 * scale).all()


# ---- paired-row fast mode: two line fetches per sample ----
@pytest.mark.parametrize("case", ["enc", "dec", "oob", "points2", "generic_k"])
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.bfloat16])
def test_pairs_mode_matches_fp32_op_on_upcast_value(case, out_dtype):
    """pack_pairs + forward_pairs == ms_deform_attn_forward(value_bf16.float()) up to fp32 summation order, incl. samples
    hanging over every edge (w_low = -1 re-based pair, zero partner at the right edge, rows -1 / H predicated off)."""
    import visionllm_b200.msda as ext
    from oracle import msda_oracle as O
    g = torch.Generator(device="cuda").manual_seed(11)
    shapes_l = [(20, 27), (10, 14), (5, 7), (3, 4)]
    L, P = {"points2": (4, 2), "generic_k": (3, 2)}.get(case, (4, 4))
    shapes_l = shapes_l[:L]
    shapes = torch.tensor(shapes_l, dtype=torch.int64, device="cuda")
    lsi = torch.cat((shapes.new_zeros(1), shapes.prod(1).cumsum(0)[:-1]))
    S = int(shapes.prod(1).sum())
    N, M, D = 3, 8, 32
    Lq = S if case != "dec" else 37
    value = torch.randn(N, S, M, D, device="cuda", generator=g).bfloat16()
    spread = 1.6 if case == "oob" else 1.05
    loc = (torch.rand(N, Lq, M, L, P, 2, device="cuda", generator=g) - 0.5) * spread + 0.5
    aw = torch.softmax(torch.randn(N, Lq, M, L * P, device="cuda", generator=g), -1).view(N, Lq, M, L, P).contiguous()
    pairs = ext.ms_deform_attn_pack_pairs(value, shapes, lsi)
    # layout contract of the pack kernel
    assert not pairs[-1].any()                      # the all-zero line off-map corners read
    pairs5 = pairs[:-1].view(N, S, M, 2, D)
    assert torch.equal(pairs5[:, :, :, 0], value)
    right = torch.zeros_like(value)
    for (H, W), st in zip(shapes_l, lsi.tolist()):
        v = value[:, st:st + H * W].view(N, H, W, M, D)
        r = torch.zeros_like(v); r[:, :, :-1] = v[:, :, 1:]
        right[:, st:st + H * W] = r.view(N, H * W, M, D)
    assert torch.equal(pairs5[:, :, :, 1], right)
    fast = ext.ms_deform_attn_forward_pairs(pairs, shapes, lsi, loc, aw, out_dtype)
    ref = ext.ms_deform_attn_forward(value.float(), shapes, lsi, loc, aw, 64)
    orc = torch.from_numpy(O.forward_kernel_semantics(value.float().cpu().numpy(), shapes.cpu().numpy(), lsi.cpu().numpy(),
                                                      loc.cpu().numpy(), aw.cpu().numpy())).cuda()
    assert fast.dtype == out_dtype and fast.shape == ref.shape
    scale = orc.abs().max().item()
    if out_dtype == torch.float32:
        assert (fast - ref).abs().max().item() <= 1e-5 * scale
        assert (fast - orc).abs().max().item() <= 1e-5 * scale
    else:
        assert ((fast.float() - ref).abs() <= 2.0 ** -8 * ref.abs() + 1e-5 * scale).all()


def test_pairs_mode_skips_out_of_map_corners_like_the_reference():
    """A corner outside the map is never read (reference .cuh:31-58): poison everything a sample at the map border must
    not touch with NaN and compare with the fp32 operator on the same poisoned value."""
    import visionllm_b200.msda as ext
    shapes = torch.tensor([[6, 5], [3, 4]], dtype=torch.int64, device="cuda")
    lsi = torch.tensor([0, 30], dtype=torch.int64, device="cuda")
    S, N, M, D, L, P = 42, 1, 2, 32, 2, 2
    g = torch.Generator(device="cuda").manual_seed(3)
    value = torch.randn(N, S, M, D, device="cuda", generator=g).bfloat16()
    value[:, 5] = float("nan")       # pixel (1, 0) of level 0: the row-wrapped "right neighbour" of pixel (0, 4)
    value[:, 29] = float("nan")      # last pixel of level 0
    # queries whose samples hang over the right / top / left borders of level 0, and far outside
    pts = torch.tensor([[[0.99, 0.05], [0.95, 0.05]], [[-0.05, 0.3], [0.3, -0.05]], [[1.15, 0.5], [0.5, 1.3]]],
                       device="cuda")                                        # [Lq = 3, P = 2, (x, y)]
    loc = pts.view(1, 3, 1, 1, 2, 2).expand(N, 3, M, L, 2, 2).contiguous()
    aw = torch.full((N, 3, M, L, P), 1.0 / (L * P), device="cuda")
    pairs = ext.ms_deform_attn_pack_pairs(value, shapes, lsi)
    fast = ext.ms_deform_attn_forward_pairs(pairs, shapes, lsi, loc, aw, torch.float32)
    ref = ext.ms_deform_attn_forward(value.float(), shapes, lsi, loc, aw, 64)
    assert torch.equal(torch.isnan(fast), torch.isnan(ref))
    ok = ~torch.isnan(ref)
    assert (fast[ok] - ref[ok]).abs().max().item() <= 1e-5


def test_pairs_mode_full_size_constant_field():
    import visionllm_b200.msda as ext
    value, shapes, lsi, loc, attw = _full_size(N=2)
    loc = loc.clamp(0.2, 0.8).contiguous()
    pairs = ext.ms_deform_attn_pack_pairs(torch.ones_like(value).bfloat16(), shapes, lsi)
    out = ext.ms_deform_attn_forward_pairs(pairs, shapes, lsi, loc, attw, torch.float32)
    assert (out - 1.0).abs().max().item() < 1e-5


def test_bf16_value_rejects_unsupported():
    import visionllm_b200.msda as ext
    shapes = torch.tensor([[4, 4]], dtype=torch.int64, device="cuda")
    lsi = torch.zeros(1, dtype=torch.int64, device="cuda")
    v = torch.zeros(1, 16, 2, 16, device="cuda", dtype=torch.bfloat16)          # D = 16: not the fast-mode shape
    loc = torch.zeros(1, 3, 2, 1, 4, 2, device="cuda"); aw = torch.zeros(1, 3, 2, 1, 4, device="cuda")
    with pytest.raises(RuntimeError):
        ext.ms_deform_attn_forward_bf16(v, shapes, lsi, loc, aw)
    with pytest.raises(RuntimeError):
        ext.ms_deform_attn_forward_bf16(v.float(), shapes, lsi, loc, aw)


@pytest.mark.skipif(__import__("os").environ.get("VLLM_EXPERIMENTAL") != "1", reason="opt-in: experimental kernel "
                    "variants not yet validated on hardware (set VLLM_EXPERIMENTAL=1)")
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.bfloat16])
def test_pairs_mode_fhfma_variant_within_bf16_weight_error(out_dtype):
    """vllm_msda_set_variant(16): per-corner weights rounded to bf16, products on FHFMA.BF16 with fp32 accumulation.
    Each term carries at most 2^-9 relative error, so the output stays within 2^-8 of sum |w_i v_i| of the exact op."""
    import visionllm_b200.msda as ext
    from visionllm_b200 import _lib
    value, shapes, lsi, loc, attw = _full_size(N=2, seed=4)
    vb = value.bfloat16()
    pairs = ext.ms_deform_attn_pack_pairs(vb, shapes, lsi)
    try:
        _lib.lib().vllm_msda_set_variant(0)
        ref = ext.ms_deform_attn_forward_pairs(pairs, shapes, lsi, loc, attw, torch.float32)
        _lib.lib().vllm_msda_set_variant(16)
        got = ext.ms_deform_attn_forward_pairs(pairs, shapes, lsi, loc, attw, out_dtype)
    finally:
        _lib.lib().vllm_msda_set_variant(0)
    bound = ext.ms_deform_attn_forward_pairs(ext.ms_deform_attn_pack_pairs(vb.abs(), shapes, lsi), shapes, lsi, loc, attw,
                                             torch.float32)                      # sum |w_i| |v_i| per output
    slack = 2.0 ** -8 * bound + (2.0 ** -8 * ref.abs() if out_dtype == torch.bfloat16 else 0) + 1e-6
    assert ((got.float() - ref).abs() <= slack).all()


# ---- the reference's OWN CUDA kernel, rebuilt for sm_100 (oracle/build_msda_ref.py), as a GPU-side oracle: its
#      results on a B200 are stored in tests/golden/msda_cuda_ref.npz (tests/golden/gen_golden_msda_cuda.py) ----
REF_CUDA_CASES = [c for c in CASES if c[3] in (32, 16)][:6]


def grad_output(shape):
    return np.random.default_rng(22).standard_normal(shape)


def sample_index(n, ci, size=2048):
    return np.sort(np.random.default_rng(1000 + ci).choice(n, min(n, size), replace=False))


@pytest.mark.parametrize("ci", range(len(REF_CUDA_CASES)),
                         ids=[f"L{len(c[0])}D{c[3]}P{c[5]}" for c in REF_CUDA_CASES])
def test_forward_matches_the_reference_cuda_kernel(golden_dir, ci):
    """ms_deform_attn_forward of the reference extension (unipose/ops/src/cuda/ms_deform_im2col_cuda.cuh, nvcc default
    -fmad=true) vs ours on the same inputs: fp32 within reassociation noise, fp64 to 1e-12; the backward too.  The
    golden holds a fixed sample of each reference result and the full result's max |x| (the tolerance scale)."""
    g = np.load(os.path.join(golden_dir, "msda_cuda_ref.npz"))
    ext = _ext()
    value, shapes, lsi, loc, attw = make_case(*REF_CUDA_CASES[ci], seed=21)
    assert np.allclose([a.astype(np.float64).sum() for a in (value, loc, attw)], g[f"c{ci}_checksum"], rtol=1e-12)
    v, sh, ls, lo, w = _dev(value, shapes, lsi, loc, attw)

    def check(name, mine, tol):
        a = mine.cpu().numpy().reshape(-1)
        assert np.abs(a[sample_index(a.size, ci)] - g[f"c{ci}_{name}"]).max() <= tol

    for flags in (0, 1):
        check("out32", ext.ms_deform_attn_forward(v, sh, ls, lo, w, 64, flags=flags),
              1e-5 * max(1.0, float(g[f"c{ci}_out32_absmax"])))
    v64, lo64, w64 = v.double(), lo.double(), w.double()
    t64 = ext.ms_deform_attn_forward(v64, sh, ls, lo64, w64, 64)
    check("out64", t64, 1e-12)
    go = torch.from_numpy(grad_output(t64.shape)).cuda()
    for name, grad in zip(("gv", "gl", "gw"), ext.ms_deform_attn_backward(v64, sh, ls, lo64, w64, go, 64)):
        check(name, grad, 1e-9 * max(1.0, float(g[f"c{ci}_{name}_absmax"])))
