"""GPU parity of the fused attention kernel against a plain PyTorch fp32 reference
(softmax in fp32 like the reference's eager paths, internlm2/modeling_internlm2.py:394).
Tolerance: bf16 P and bf16 output rounding -> |out - ref| <= 2^-7*|ref| + 2e-3*max|ref|."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def ref_attn(q, k, v, causal, seqlens=None):
    B, Tq, H, D = q.shape
    Tk, Hkv = k.shape[1], k.shape[2]
    qf = q.float().permute(0, 2, 1, 3)
    kf = k.float().permute(0, 2, 1, 3).repeat_interleave(H // Hkv, 1)
    vf = v.float().permute(0, 2, 1, 3).repeat_interleave(H // Hkv, 1)
    s = qf @ kf.transpose(-1, -2) * D ** -0.5
    if causal:
        i = torch.arange(Tq, device=q.device)[:, None] + (Tk - Tq)
        j = torch.arange(Tk, device=q.device)[None, :]
        s = s.masked_fill(j > i, float("-inf"))
    if seqlens is not None:
        j = torch.arange(Tk, device=q.device)[None, None, None, :]
        s = s.masked_fill(j >= seqlens[:, None, None, None], float("-inf"))
    o = torch.softmax(s, -1) @ vf
    o = o.permute(0, 2, 1, 3).reshape(B, Tq, H * D)
    return o


@pytest.fixture(params=[0, 1, 2], ids=["tcgen05_tc2", "warp_mma", "tcgen05_pingpong"])
def variant(request):
    """Run every case on the tcgen05/TMEM kernel (head_dim 128) and on the warp-MMA kernel."""
    from visionllm_b200 import _lib
    _lib.lib().vllm_attention_set_variant(request.param)
    yield request.param
    _lib.lib().vllm_attention_set_variant(0)


def check(out, ref):
    tol = ref.abs() * 2.0 ** -7 + 2e-3 * ref.abs().max()
    bad = (out.float() - ref).abs() > tol
    assert not bad.any(), f"{int(bad.sum())}/{bad.numel()} off, max {(out.float() - ref).abs().max().item()}"


@pytest.mark.parametrize("B,T,H,D,causal", [
    (2, 1025, 5, 128, False),     # InternViT tile: 1025 = 16*64 + 1 (ragged last tile)
    (1, 577, 4, 64, False),       # CLIP-L tile
    (2, 300, 8, 32, False),       # GDINO-size heads
    (2, 1536, 4, 128, True),      # LLM causal
    (1, 64, 2, 128, True),
    (1, 1, 2, 128, True),
    (3, 130, 3, 128, True),
    (2, 257, 2, 128, False),      # one key past two KV tiles, one row past the first CTA
    (1, 3136, 2, 128, True),      # released-7B sequence length
])
def test_attention_packed_qkv(B, T, H, D, causal, variant):
    from visionllm_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(T)
    qkv = torch.randn(B, T, 3, H, D, device="cuda", generator=g).bfloat16()
    q, k, v = qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2]       # strided views, no copies
    out = ops.attention(q, k, v, causal=causal)
    check(out, ref_attn(q, k, v, causal))


def test_attention_gqa_and_seqlens_and_cross(variant):
    from visionllm_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(1)
    B, Tq, Tk, H, Hkv, D = 3, 200, 333, 8, 2, 128
    q = torch.randn(B, Tq, H, D, device="cuda", generator=g).bfloat16()
    k = torch.randn(B, Tk, Hkv, D, device="cuda", generator=g).bfloat16()
    v = torch.randn(B, Tk, Hkv, D, device="cuda", generator=g).bfloat16()
    check(ops.attention(q, k, v), ref_attn(q, k, v, False))
    check(ops.attention(q, k, v, causal=True), ref_attn(q, k, v, True))
    sl = torch.tensor([333, 17, 150], dtype=torch.int32, device="cuda")
    check(ops.attention(q, k, v, seqlens=sl), ref_attn(q, k, v, False, sl))


def test_attention_large_magnitude_is_stable(variant):
    from visionllm_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(2)
    q = (torch.randn(1, 256, 2, 128, device="cuda", generator=g) * 8).bfloat16()
    k = (torch.randn(1, 256, 2, 128, device="cuda", generator=g) * 8).bfloat16()
    v = torch.randn(1, 256, 2, 128, device="cuda", generator=g).bfloat16()
    out = ops.attention(q, k, v)
    assert torch.isfinite(out.float()).all()
    check(out, ref_attn(q, k, v, False))


def test_attention_head_dim_256_and_key_mask():
    """GDINO bi-attention shapes: head_dim 256, arbitrary key_padding_mask (padded pixels are not a suffix)."""
    from visionllm_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(9)
    B, Tq, Tk, H, D = 2, 70, 333, 4, 256
    q = torch.randn(B, Tq, H, D, device="cuda", generator=g).bfloat16()
    k = torch.randn(B, Tk, H, D, device="cuda", generator=g).bfloat16()
    v = torch.randn(B, Tk, H, D, device="cuda", generator=g).bfloat16()
    km = torch.rand(B, Tk, device="cuda", generator=g) > 0.3
    km[:, 0] = True
    out = ops.attention(q, k, v, key_mask=km)
    s = (q.float().permute(0, 2, 1, 3) @ k.float().permute(0, 2, 3, 1)) * D ** -0.5
    s = s.masked_fill(~km[:, None, None, :], float("-inf"))
    ref = (torch.softmax(s, -1) @ v.float().permute(0, 2, 1, 3)).permute(0, 2, 1, 3).reshape(B, Tq, H * D)
    check(out, ref)
    # head_dim 128 with a key mask: tcgen05 kernel with the mask operand (r2)
    q2, k2, v2 = q[..., :128].contiguous(), k[..., :128].contiguous(), v[..., :128].contiguous()
    out2 = ops.attention(q2, k2, v2, key_mask=km)
    s2 = (q2.float().permute(0, 2, 1, 3) @ k2.float().permute(0, 2, 3, 1)) * 128 ** -0.5
    s2 = s2.masked_fill(~km[:, None, None, :], float("-inf"))
    ref2 = (torch.softmax(s2, -1) @ v2.float().permute(0, 2, 1, 3)).permute(0, 2, 1, 3).reshape(B, Tq, H * 128)
    check(out2, ref2)


def test_attention_full_attn_mask():
    """nn.MultiheadAttention-style [B*H, Tq, Tk] boolean mask (True = attend here), head_dim 64."""
    from visionllm_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(10)
    B, T, H, D = 2, 37, 4, 64
    q = torch.randn(B, T, H, D, device="cuda", generator=g).bfloat16()
    k = torch.randn(B, T, H, D, device="cuda", generator=g).bfloat16()
    v = torch.randn(B, T, H, D, device="cuda", generator=g).bfloat16()
    am = torch.rand(B * H, T, T, device="cuda", generator=g) > 0.4
    am |= torch.eye(T, device="cuda", dtype=torch.bool)[None]
    out = ops.attention(q, k, v, attn_mask=am)
    s = (q.float().permute(0, 2, 1, 3) @ k.float().permute(0, 2, 3, 1)) * D ** -0.5
    s = s.masked_fill(~am.view(B, H, T, T), float("-inf"))
    ref = (torch.softmax(s, -1) @ v.float().permute(0, 2, 1, 3)).permute(0, 2, 1, 3).reshape(B, T, H * D)
    check(out, ref)


@pytest.mark.parametrize("D,H", [(256, 4), (64, 4), (32, 8)])
def test_attention_split_kv_few_queries_many_keys(D, H):
    """GDINO text->vision shape class: a handful of queries over thousands of keys -> the key axis is split across
    CTAs and merged (vllm_attention_bf16 workspace path); with and without a key mask."""
    from visionllm_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(D)
    B, Tq, Tk = 2, 80, 5000
    q = torch.randn(B, Tq, H, D, device="cuda", generator=g).bfloat16()
    k = torch.randn(B, Tk, H, D, device="cuda", generator=g).bfloat16()
    v = torch.randn(B, Tk, H, D, device="cuda", generator=g).bfloat16()
    km = torch.rand(B, Tk, device="cuda", generator=g) > 0.2
    for mask in (None, km):
        out = ops.attention(q, k, v, key_mask=mask)
        s_ = (q.float().permute(0, 2, 1, 3) @ k.float().permute(0, 2, 3, 1)) * D ** -0.5
        if mask is not None:
            s_ = s_.masked_fill(~mask[:, None, None, :], float("-inf"))
        ref = (torch.softmax(s_, -1) @ v.float().permute(0, 2, 1, 3)).permute(0, 2, 1, 3).reshape(B, Tq, H * D)
        check(out, ref)


@pytest.mark.parametrize("D", [128, 256])
@pytest.mark.parametrize("Tq,Tk", [(300, 80), (80, 4352), (257, 640), (1500, 96)])
def test_attention_tcgen05_key_mask_and_split_kv(D, Tq, Tk):
    """r2: head_dim 256 and key-masked head_dim 128 calls run on the tcgen05 kernel (attention_tc2.cu<D, KM>): the
    GDINO bi-attention's two shapes (many vision queries x 80 text keys; 80 text queries x thousands of vision keys,
    split along the key axis) with arbitrary key masks -- 16-byte mask loads (Tk % 16 == 0), fully masked 64-key tiles,
    a batch entry whose mask leaves a single key.  Checked against fp32 torch and against the warp-MMA kernel."""
    from visionllm_b200 import _lib, ops
    g = torch.Generator(device="cuda").manual_seed(D + Tq + Tk)
    B, H = 3, 4
    q = torch.randn(B, Tq, H, D, device="cuda", generator=g).bfloat16()
    k = torch.randn(B, Tk, H, D, device="cuda", generator=g).bfloat16()
    v = torch.randn(B, Tk, H, D, device="cuda", generator=g).bfloat16()
    km = torch.rand(B, Tk, device="cuda", generator=g) > 0.3
    km[0, :] = True
    if Tk >= 256:
        km[1, 64:192] = False                              # two whole key tiles masked out
    km[2, :] = False
    km[2, Tk // 2] = True                                  # one key left
    for mask in (km, None):
        out = ops.attention(q, k, v, key_mask=mask)
        s_ = (q.float().permute(0, 2, 1, 3) @ k.float().permute(0, 2, 3, 1)) * D ** -0.5
        if mask is not None:
            s_ = s_.masked_fill(~mask[:, None, None, :], float("-inf"))
        ref = (torch.softmax(s_, -1) @ v.float().permute(0, 2, 1, 3)).permute(0, 2, 1, 3).reshape(B, Tq, H * D)
        check(out, ref)
        _lib.lib().vllm_attention_set_variant(1)
        try:
            warp = ops.attention(q, k, v, key_mask=mask)
        finally:
            _lib.lib().vllm_attention_set_variant(0)
        check(out, warp.float())


@pytest.mark.parametrize("B,H,T,D,group", [(2, 8, 690, 32, 69), (1, 4, 200, 64, 40), (2, 2, 333, 128, 111), (1, 8, 3450, 32, 69)])
def test_live_tile_lists_give_the_dense_result(B, H, T, D, group):
    """vllm_attention_mask_tiles + vllm_attention_bf16_tiles (UniPose's keypoint decoder mask: groups of 1 + 68 queries that
    attend within their group plus a few stripes): the tile lists match a torch evaluation of "any allowed pair per 64 x 64
    tile", and walking only the live tiles reproduces the dense walk bit for bit -- including query rows that may attend
    nothing (zero output) and query blocks with no live tile at all."""
    from visionllm_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(T + D)
    q, k, v = (torch.randn(B, T, H, D, device="cuda", generator=g).bfloat16() for _ in range(3))
    idx = torch.arange(T, device="cuda")
    allow = (idx[:, None] // group) == (idx[None, :] // group)                       # block diagonal
    allow = allow[None].repeat(B * H, 1, 1)
    n_groups = (T + group - 1) // group
    for bh in range(B * H):                                                            # a few off-diagonal stripes per (batch, head)
        for _ in range(2):
            gi, gj = (int(x) for x in torch.randint(0, n_groups, (2,), device="cuda", generator=g))
            allow[bh, gi * group:(gi + 1) * group, gj * group] = True
    allow[0, 5] = False                                                                # a query row that attends nothing
    if T > 128:
        allow[-1, 64:128] = False                                                      # a whole query block without live tiles
    dense = ops.attention(q, k, v, attn_mask=allow)
    tiles = ops.attention_mask_tiles(allow)
    nqb = nkt = (T + 63) // 64
    pad = nqb * 64 - T
    ap = torch.nn.functional.pad(allow, (0, pad, 0, pad))
    any_t = ap.view(B * H, nqb, 64, nkt, 64).any(4).any(2)                             # [BH, nqb, nkt]
    assert torch.equal(tiles.counts.long(), any_t.sum(-1))
    for bh in range(0, B * H, max(1, B * H // 3)):
        for qb in range(0, nqb, max(1, nqb // 4)):
            n = int(tiles.counts[bh, qb])
            assert tiles.lists[bh, qb, :n].tolist() == torch.nonzero(any_t[bh, qb]).flatten().tolist()
    sparse = ops.attention(q, k, v, attn_mask=tiles)
    assert torch.equal(sparse, dense)
    assert not sparse[0, 5, :D].any()                                                  # head 0 of batch 0: the empty row
    if T >= 600:
        assert float(any_t.float().mean()) < 0.5                                       # the point: most tiles are skipped
    ref_s = (q.float().permute(0, 2, 1, 3) @ k.float().permute(0, 2, 3, 1)) * D ** -0.5
    ref_s = ref_s.masked_fill(~allow.view(B, H, T, T), float("-inf"))
    p = torch.softmax(ref_s, -1).nan_to_num(0.0)
    ref = (p @ v.float().permute(0, 2, 1, 3)).permute(0, 2, 1, 3).reshape(B, T, H * D)
    assert ((sparse.float() - ref).norm() / ref.norm()).item() < 6e-3


@pytest.mark.parametrize("causal", [True, False])
def test_attention_is_reproducible_at_the_llm_shape(causal):
    """The same inputs give bit-identical outputs on every call, at the Vicuna-7B shape of the flagship forward (8 x 1536
    tokens, 32 heads of 128, q/k/v slices of one packed qkv tensor).  Before the epilogue waited on a barrier committed
    after the last P V product, tc2 warps could read O from tensor memory early and a few 32-row groups changed between
    calls."""
    from visionllm_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(0)
    B, T, H, D = 8, 1536, 32, 128
    qkv = torch.randn(B, T, 3 * H * D, device="cuda", generator=g).bfloat16()
    q, k, v = (qkv[..., i * H * D:(i + 1) * H * D].unflatten(-1, (H, D)) for i in range(3))
    first = ops.attention(q, k, v, causal=causal)
    for _ in range(4):
        assert torch.equal(ops.attention(q, k, v, causal=causal), first)
