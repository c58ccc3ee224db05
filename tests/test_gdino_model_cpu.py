"""CPU: the whole Grounding-DINO stage -- backbone, neck, encoder, mask FPN, two-stage selection, decoder, heads -- of
`visionllm_b200.gdino_model.B200GroundingDinoForObjectDetection` against the REFERENCE'S OWN
`OVGroundingDinoForObjectDetection.forward_test` run on CPU in fp32 with the same state dict, stored in
tests/golden/gdino_{stage,internimage,neck}_cpu.npz (tests/golden/gen_golden_gdino_cpu.py, which takes its
configurations, seeds and inputs from this file).  Kernels are replaced by fp32 torch stand-ins in this test only (no
GPU here); this pins the host logic: layouts, masks, valid ratios, reference points, top-k selection, box refinement,
head wiring, parameter names."""
import json
import os
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
from test_gdino_logic_cpu import torch_kernels  # noqa: E402,F401  (fixture)

SWIN_VARIANTS = {"swin24": (11, False), "swin32": (11, True)}        # tag: (weight seed, B200 Swin backbone)
STAGE_CASES = [("swin24", False), ("swin24", True), ("swin32", True)]  # (variant, ragged pixel mask)
NECK_SEED, INTERNIMAGE_SEED = 12, 21


def swin_config_kwargs(b200_backbone):
    from transformers import SwinConfig
    bc = SwinConfig(image_size=64, embed_dim=32 if b200_backbone else 24, depths=[1, 2, 1, 1], num_heads=[1, 2, 4, 8],
                    window_size=4, out_features=["stage1", "stage2", "stage3", "stage4"])
    return dict(backbone_config=bc, d_model=256, encoder_layers=2, decoder_layers=2, encoder_ffn_dim=256,
                decoder_ffn_dim=256, num_queries=20, num_feature_levels=4, dropout=0., attention_dropout=0.,
                activation_dropout=0., fusion_dropout=0., fusion_droppath=0., text_enhancer_dropout=0.,
                disable_custom_kernels=True, mask_dim=256, norm="GN", l_hidden_size=64)


def internimage_config_kwargs():
    # H width (the reference hard-codes the neck's input widths to 320..2560, gd.py:5183), one layer per level
    bc = dict(model_type="internimage-H", core_op="DCNv3_pytorch", depths=[1, 1, 1, 1], level2_post_norm_block_ids=[0],
              with_cp=False)
    return dict(backbone_config=bc, d_model=256, encoder_layers=1, decoder_layers=1, encoder_ffn_dim=256,
                decoder_ffn_dim=256, num_queries=12, num_feature_levels=4, dropout=0., attention_dropout=0.,
                activation_dropout=0., fusion_dropout=0., fusion_droppath=0., text_enhancer_dropout=0.,
                disable_custom_kernels=True, mask_dim=256, norm="GN", l_hidden_size=64)


def case_name(tag, ragged):
    return f"{tag}_{'ragged' if ragged else 'full'}"


def checksum(*ts):
    return np.array([float(t.double().sum()) for t in ts])


def gated(sd):
    for k in sd:                                                  # LayerScale-style gates: make the fusion path count
        if k.endswith("vision_param") or k.endswith("text_param"):
            sd[k] = sd[k] * 0 + 0.5
    return sd


def stage_inputs(ragged, l_hidden):
    g = torch.Generator().manual_seed(5)
    B, Hh, W = 2, 128, 160
    x = torch.randn(B, 3, Hh, W, generator=g)
    pm = torch.ones(B, Hh, W, dtype=torch.long)
    if ragged:
        pm[1, 96:, :] = 0
        pm[1, :, 120:] = 0
    tq = torch.randn(B, 5, 4, l_hidden, generator=g)
    tm = torch.ones(B, 5, dtype=torch.bool)
    tm[1, 3:] = False
    return x, pm, tq, tm


def neck_inputs(l_hidden):
    g = torch.Generator().manual_seed(13)
    x = torch.randn(1, 3, 100, 136, generator=g)
    pm = torch.ones(1, 100, 136, dtype=torch.long)
    pm[0, 80:] = 0
    return x, pm, torch.randn(1, 3, 4, l_hidden, generator=g), torch.ones(1, 3, dtype=torch.bool)


def internimage_inputs(l_hidden):
    g = torch.Generator().manual_seed(6)
    B, Hh, W = 2, 64, 96
    x = torch.randn(B, 3, Hh, W, generator=g)
    pm = torch.ones(B, Hh, W, dtype=torch.long)
    pm[1, 32:, :] = 0
    return x, pm, torch.randn(B, 4, 4, l_hidden, generator=g), torch.ones(B, 4, dtype=torch.bool)


def reference_config(config_json):
    """The reference GroundingDinoConfig's attributes as the generator recorded them (a Swin backbone config is
    rebuilt as transformers' SwinConfig; the InternImage one stays the dict the reference keeps)."""
    from transformers import SwinConfig
    d = json.loads(config_json)
    bc = d.get("backbone_config")
    if isinstance(bc, dict) and bc.get("model_type") == "swin":
        d["backbone_config"] = SwinConfig.from_dict(bc)
    return SimpleNamespace(**d)


def build_ours(g, tag, seed, b200_backbone=False):
    from weights_util import key_shapes, seeded_state_dict
    from visionllm_b200.gdino_model import B200GroundingDinoForObjectDetection
    from visionllm_b200.swin import B200SwinBackbone
    cfg = reference_config(str(g[f"{tag}_config"]))
    bb = B200SwinBackbone(cfg.backbone_config) if b200_backbone else None
    ours = B200GroundingDinoForObjectDetection(cfg, backbone_model=bb).eval()
    # identical parameter names: the reference's state-dict keys and shapes, as recorded
    assert [list(k) for k in key_shapes(ours)] == json.loads(str(g[f"{tag}_keys"]))
    ours.load_state_dict(gated(seeded_state_dict(ours, seed)), strict=True)
    return cfg, ours


def assert_stage_outputs(g, name, b):
    a_logits, a_boxes, a_masks = (torch.from_numpy(g[f"{name}_{k}"]) for k in ("logits", "pred_boxes", "pred_masks"))
    assert a_logits.shape == b.logits.shape and a_masks.shape == b.pred_masks.shape
    finite = torch.isfinite(a_logits)
    assert torch.equal(finite, torch.isfinite(b.logits))                      # -inf padding pattern identical
    assert (a_logits[finite] - b.logits[finite]).abs().max() < 2e-3
    assert (a_boxes - b.pred_boxes).abs().max() < 1e-4
    assert (a_masks - b.pred_masks).abs().max() < 2e-2 * a_masks.abs().max().clamp(min=1)


@pytest.fixture()
def gn_kernel(monkeypatch, torch_kernels):  # noqa: F811
    import visionllm_b200.ops as ops

    from oracle import torch_kernels as TK

    monkeypatch.setattr(ops, "groupnorm_nhwc", TK.groupnorm_nhwc)
    monkeypatch.setattr(ops, "conv2d_s1_rows", TK.conv2d_s1_rows)
    monkeypatch.setattr(ops, "upsample_add_nhwc", TK.upsample_add_nhwc)


@pytest.mark.parametrize("ragged,b200_backbone", [(False, False), (True, False), (True, True)])
def test_whole_stage_matches_reference_forward_test(golden_dir, gn_kernel, ragged, b200_backbone):
    g = np.load(os.path.join(golden_dir, "gdino_stage_cpu.npz"))
    tag = "swin32" if b200_backbone else "swin24"
    cfg, ours = build_ours(g, tag, SWIN_VARIANTS[tag][0], b200_backbone)
    x, pm, tq, tm = stage_inputs(ragged, cfg.l_hidden_size)
    name = case_name(tag, ragged)
    assert np.allclose(checksum(x, tq), g[f"{name}_checksum"], rtol=1e-12)
    with torch.no_grad():
        b = ours.forward_test(x, pixel_mask=pm, text_query=tq, text_query_masks=tm)
    assert_stage_outputs(g, name, b)


def test_neck_integer_outputs_match_reference(golden_dir, gn_kernel):
    """spatial_shapes / level_start_index (int64) exactly; valid_ratios, masks exactly (same torch ops); the float maps
    on every 4th token row."""
    n = np.load(os.path.join(golden_dir, "gdino_neck_cpu.npz"))
    g = np.load(os.path.join(golden_dir, "gdino_stage_cpu.npz"))
    cfg, ours = build_ours(g, "swin24", NECK_SEED)
    x, pm, tq, tm = neck_inputs(cfg.l_hidden_size)
    assert np.allclose(checksum(x, tq), n["checksum"], rtol=1e-12)
    with torch.no_grad():
        feats = ours.model.backbone_features(x)
        src, mflat, pos, shapes, lsi, vr = ours.model.neck(feats, pm)
    assert torch.equal(shapes, torch.from_numpy(n["spatial_shapes"])) and shapes.dtype == torch.int64
    assert torch.equal(lsi, torch.from_numpy(n["level_start_index"]))
    assert torch.equal(~mflat, torch.from_numpy(n["vision_attention_mask"]))
    assert torch.equal(vr, torch.from_numpy(n["valid_ratios"]))
    assert (src[:, ::4] - torch.from_numpy(n["vision_features_sub"])).abs().max() < 1e-4
    assert (pos[:, ::4] - torch.from_numpy(n["vision_position_embedding_sub"])).abs().max() < 1e-5


def test_whole_stage_with_internimage_backbone_matches_reference(golden_dir, gn_kernel, monkeypatch):
    """`backbone_config = {'model_type': 'internimage-H', ...}` (gd.py:2073-2074, 5154-5195): the reference builds
    `GroundingDinoInternImageBackbone`, we build `visionllm_b200.internimage` from the same dict; same state dict, same
    forward_test outputs.  The reference runs its pure-PyTorch core op; ours runs the C oracle of the CUDA core."""
    import visionllm_b200.dcnv3 as dcn
    import visionllm_b200.ops as ops
    from oracle import dcnv3_oracle as O

    def layernorm(x, w, b, eps, out=None, gelu=False, residual=None):
        y = F.layer_norm(x.float(), (x.shape[-1],), w.float(), b.float(), eps)
        if residual is not None:
            y = y + residual.float()
        return F.gelu(y) if gelu else y

    def dwconv_nhwc(x, wt, bias, k):
        C = x.shape[-1]
        return F.conv2d(x.float().permute(0, 3, 1, 2), wt.float().t().reshape(C, 1, k, k), bias.float(), padding=k // 2,
                        groups=C).permute(0, 2, 3, 1).contiguous()

    def dcnv3_prep(packed, G, K, with_scale):
        lead = packed.shape[:-1]
        mask = F.softmax(packed[..., G * K * 2:G * K * 3].reshape(*lead, G, K), -1).reshape(*lead, G * K).contiguous()
        return (packed[..., :G * K * 2].contiguous(), mask,
                packed[..., G * K * 3:G * K * 3 + G].sigmoid() if with_scale else None)

    def dcnv3_blend(core, xproj, scale, gc):
        if scale is None:
            return core
        s_ = scale[..., None].expand(*scale.shape, gc).reshape(core.shape)
        return core * (1 - s_) + xproj * s_

    def dcnv3_forward(inp, offset, mask, kh, kw, sh, sw, ph, pw, dh, dw, group, gc, offset_scale, step=256, **kw_):
        return torch.from_numpy(np.asarray(O.forward(inp.float().numpy(), offset.float().numpy(), mask.float().numpy(),
                                                     kh, kw, sh, sw, ph, pw, dh, dw, group, gc, offset_scale),
                                           dtype=np.float32))

    for name, fn in (("layernorm", layernorm), ("dwconv_nhwc", dwconv_nhwc),
                     ("dcnv3_prep", dcnv3_prep), ("dcnv3_blend", dcnv3_blend)):
        monkeypatch.setattr(ops, name, fn)
    monkeypatch.setattr(dcn, "dcnv3_forward", dcnv3_forward)

    g = np.load(os.path.join(golden_dir, "gdino_internimage_cpu.npz"))
    cfg, ours = build_ours(g, "internimage", INTERNIMAGE_SEED)
    assert type(ours.model.backbone.conv_encoder.model).__name__ == "B200InternImage"
    x, pm, tq, tm = internimage_inputs(cfg.l_hidden_size)
    assert np.allclose(checksum(x, tq), g["internimage_checksum"], rtol=1e-12)
    with torch.no_grad():
        b = ours.forward_test(x, pixel_mask=pm, text_query=tq, text_query_masks=tm)
    assert_stage_outputs(g, "internimage", b)


def test_conv_rows_prepadded_forms_agree(gn_kernel):
    """conv_rows / NormConv2d.rows on the zero-bordered map `upsample_add_nhwc(..., pad=)` writes (the copy-free mask-FPN chain)
    equal the plain call on the unpadded map -- for the implicit-GEMM 3x3 form (border consumed by the convolution) and for
    shapes that take the general path (border dropped again)."""
    import torch.nn as nn
    from visionllm_b200.gdino_model import NormConv2d, conv_rows
    g = torch.Generator().manual_seed(3)
    for C, k, p in ((64, 3, 1), (24, 3, 1), (64, 1, 0)):                 # 3 * 64 % 64 == 0: implicit; 3 * 24: general; 1x1
        x = torch.randn(2, 6, 7, C, generator=g)
        conv = NormConv2d(C, 32, k, padding=p, relu=True).eval()
        nn.init.normal_(conv.weight, std=0.1)
        xp = torch.nn.functional.pad(x, (0, 0, p, p, p, p))
        a, Ha, Wa = conv_rows(x, conv)
        b, Hb, Wb = conv_rows(xp, conv, prepadded=p > 0)
        assert (Ha, Wa) == (Hb, Wb) == (6, 7) and torch.allclose(a, b.reshape(a.shape), atol=1e-6)
        ra, _, _ = conv.rows(x)
        rb, _, _ = conv.rows(xp, prepadded=p > 0)
        assert ra.shape == rb.shape == (2, 42, 32) and torch.allclose(ra, rb, atol=1e-5)
