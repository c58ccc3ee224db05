"""Golden vectors for tests/test_gdino_model_cpu.py and tests/test_dropin_reference_cpu.py from the REFERENCE's own
Grounding-DINO code run on CPU in fp32 (needs the reference checkout; see ref_shim.py).

  gdino_stage_cpu.npz     `OVGroundingDinoForObjectDetection.forward_test` outputs (logits, boxes, masks) of the whole
                          stage for the Swin configurations, with the reference config's attributes (JSON) and
                          state-dict keys
  gdino_internimage_cpu.npz  the same for the InternImage-H backbone configuration
  gdino_neck_cpu.npz      what the reference's neck hands to its encoder (every 4th token row of the float maps)
  gdino_dropin_enc.npz    every call the reference's `GroundingDinoEncoder` loop makes to its layers: the keyword
                          arguments and the outputs
  gdino_dropin_dec.npz    the same for `GroundingDinoDecoder`: decoder layers, query-position head, box heads

Weights come from weights_util.seeded_state_dict (keyed by the recorded names), inputs from torch generators with the
seeds the tests use; each file records a checksum of the inputs.

    python tests/golden/gen_golden_gdino_cpu.py
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [HERE, ROOT, os.path.join(ROOT, "tests")]
import ref_shim  # noqa: E402
from weights_util import key_shapes, seeded_state_dict  # noqa: E402

import test_gdino_model_cpu as TM  # noqa: E402

SUB = 4
DROPIN_LEVELS = [(8, 10), (4, 5), (2, 3), (1, 2)]


def config_json(cfg):
    out = {}
    for k, v in vars(cfg).items():
        if k == "backbone_config":
            out[k] = v.to_dict() if hasattr(v, "to_dict") else v
            continue
        try:
            json.dumps(v)
        except TypeError:
            continue
        out[k] = v
    return json.dumps(out, sort_keys=True)


def ref_stage(gd, cfg, seed):
    ref = gd.OVGroundingDinoForObjectDetection(cfg).eval()
    ref.load_state_dict(TM.gated(seeded_state_dict(ref, seed)))
    return ref


def stage_goldens(cfgm, gd):
    out = {}
    for tag, (seed, b200_backbone) in TM.SWIN_VARIANTS.items():
        cfg = cfgm.GroundingDinoConfig(**TM.swin_config_kwargs(b200_backbone))
        ref = ref_stage(gd, cfg, seed)
        cfg.activation_function = "relu"
        out[f"{tag}_config"] = config_json(cfg)
        out[f"{tag}_keys"] = json.dumps([list(k) for k in key_shapes(ref)])
        for ragged in (False, True):
            if (tag, ragged) not in TM.STAGE_CASES:
                continue
            x, pm, tq, tm = TM.stage_inputs(ragged, cfg.l_hidden_size)
            with torch.no_grad():
                a = ref.forward_test(pixel_values=x, pixel_mask=pm, text_query=tq, text_query_masks=tm, return_dict=True)
            name = TM.case_name(tag, ragged)
            out[f"{name}_checksum"] = TM.checksum(x, tq)
            out[f"{name}_logits"] = a.logits.numpy()
            out[f"{name}_pred_boxes"] = a.pred_boxes.numpy()
            out[f"{name}_pred_masks"] = a.pred_masks.numpy()
    return out


def internimage_goldens():
    out = {}
    cfgm, gd = ref_shim.load_gdino_with_dcnv3()
    cfg = cfgm.GroundingDinoConfig(**TM.internimage_config_kwargs())
    ref = ref_stage(gd, cfg, TM.INTERNIMAGE_SEED)
    cfg.activation_function = "relu"
    out["internimage_config"] = config_json(cfg)
    out["internimage_keys"] = json.dumps([list(k) for k in key_shapes(ref)])
    x, pm, tq, tm = TM.internimage_inputs(cfg.l_hidden_size)
    with torch.no_grad():
        a = ref.forward_test(pixel_values=x, pixel_mask=pm, text_query=tq, text_query_masks=tm, return_dict=True)
    out["internimage_checksum"] = TM.checksum(x, tq)
    out["internimage_logits"] = a.logits.numpy()
    out["internimage_pred_boxes"] = a.pred_boxes.numpy()
    out["internimage_pred_masks"] = a.pred_masks.numpy()
    return out


def neck_golden(cfgm, gd):
    cfg = cfgm.GroundingDinoConfig(**TM.swin_config_kwargs(False))
    ref = ref_stage(gd, cfg, TM.NECK_SEED)
    x, pm, tq, tm = TM.neck_inputs(cfg.l_hidden_size)
    cap = {}
    orig = ref.model.encoder.forward

    def spy(**kw):
        cap.update(kw)
        return orig(**kw)

    ref.model.encoder.forward = spy
    with torch.no_grad():
        ref.forward_test(pixel_values=x, pixel_mask=pm, text_query=tq, text_query_masks=tm, return_dict=True)
    return {"checksum": TM.checksum(x, tq), "spatial_shapes": cap["spatial_shapes"].numpy(),
            "level_start_index": cap["level_start_index"].numpy(),
            "vision_attention_mask": cap["vision_attention_mask"].numpy(), "valid_ratios": cap["valid_ratios"].numpy(),
            "vision_features_sub": cap["vision_features"][:, ::SUB].numpy(),
            "vision_position_embedding_sub": cap["vision_position_embedding"][:, ::SUB].numpy()}


class Recorder:
    """Forward hooks that record every call of the given modules: tensor keyword/positional arguments (stored once per
    distinct tensor object), the other arguments as JSON, and the outputs."""

    def __init__(self):
        self.arrays, self.calls, self._seen = {}, [], []

    def _tensor(self, t):
        for obj, key in self._seen:
            if obj is t:
                return key
        key = f"t{len(self._seen)}"
        self._seen.append((t, key))
        self.arrays[key] = t.detach().numpy()
        return key

    def _encode(self, v):
        if isinstance(v, torch.Tensor):
            return {"tensor": self._tensor(v)}
        if isinstance(v, (tuple, list)):
            return {"seq": [self._encode(x) for x in v]}
        return {"value": v}

    def watch(self, name, module):
        def hook(mod, args, kwargs, output):
            self.calls.append({"module": name, "args": [self._encode(a) for a in args],
                               "kwargs": {k: self._encode(v) for k, v in kwargs.items()}, "output": self._encode(output)})
        module.register_forward_hook(hook, with_kwargs=True)

    def save(self, path, **extra):
        np.savez(path, calls=json.dumps(self.calls), **self.arrays, **extra)


def _levels():
    shapes = torch.tensor(DROPIN_LEVELS)
    return shapes, torch.cat((shapes.new_zeros(1), shapes.prod(1).cumsum(0)[:-1])), int(shapes.prod(1).sum())


def dropin_encoder(cfgm, gd, seed=77):
    cfg = cfgm.GroundingDinoConfig(d_model=256, encoder_layers=2, encoder_attention_heads=8, encoder_ffn_dim=512,
                                   num_feature_levels=4, encoder_n_points=4, dropout=0.0, attention_dropout=0.0,
                                   activation_dropout=0.0, fusion_dropout=0.0, fusion_droppath=0.0,
                                   text_enhancer_dropout=0.0, disable_custom_kernels=True)
    enc = gd.GroundingDinoEncoder(cfg).eval()
    enc.load_state_dict(seeded_state_dict(enc, seed))
    cfg.activation_function = "relu"
    rec = Recorder()
    for i, layer in enumerate(enc.layers):
        rec.watch(f"layers.{i}", layer)
    shapes, lsi, S = _levels()
    B, T = 1, 6
    g = torch.Generator().manual_seed(1)
    src, pos, text = (torch.randn(B, S, 256, generator=g), torch.randn(B, S, 256, generator=g) * 0.5,
                      torch.randn(B, T, 256, generator=g))
    tq = torch.ones(B, T, dtype=torch.bool); tq[0, 4:] = False
    tsa, pids = gd.generate_masks_with_text_query_masks(tq)
    with torch.no_grad():
        enc(vision_features=src, vision_attention_mask=torch.zeros(B, S, dtype=torch.bool), vision_position_embedding=pos,
            spatial_shapes=shapes, level_start_index=lsi, valid_ratios=torch.ones(B, 4, 2), text_features=text,
            text_attention_mask=~tq, text_position_embedding=None, text_self_attention_masks=tsa, text_position_ids=pids,
            output_attentions=False, output_hidden_states=False, return_dict=True)
    return rec, {"keys": json.dumps([list(k) for k in key_shapes(enc)]), "seed": seed, "config": config_json(cfg)}


def dropin_decoder(cfgm, gd, seed=88):
    cfg = cfgm.GroundingDinoConfig(d_model=256, decoder_layers=2, decoder_attention_heads=8, decoder_ffn_dim=512,
                                   num_feature_levels=4, decoder_n_points=4, dropout=0.0, attention_dropout=0.0,
                                   activation_dropout=0.0, disable_custom_kernels=True)
    dec = gd.GroundingDinoDecoder(cfg).eval()
    # OVGroundingDinoForObjectDetection shares one bbox head per layer with the decoder (gd.py:2640-2652)
    dec.bbox_embed = torch.nn.ModuleList([gd.GroundingDinoMLPPredictionHead(256, 256, 4, 3) for _ in range(2)])
    dec.load_state_dict(seeded_state_dict(dec, seed))
    cfg.activation_function = "relu"
    rec = Recorder()
    for i, layer in enumerate(dec.layers):
        rec.watch(f"layers.{i}", layer)
        rec.watch(f"bbox_embed.{i}", dec.bbox_embed[i])
    rec.watch("reference_points_head", dec.reference_points_head)
    shapes, lsi, S = _levels()
    B, Q, T = 2, 9, 5
    g = torch.Generator().manual_seed(2)
    with torch.no_grad():
        dec(inputs_embeds=torch.randn(B, Q, 256, generator=g), vision_encoder_hidden_states=torch.randn(B, S, 256, generator=g),
            mask_features=None, vision_encoder_attention_mask=torch.ones(B, S, dtype=torch.bool),
            text_encoder_hidden_states=torch.randn(B, T, 256, generator=g),
            text_encoder_attention_mask=torch.tensor([[False] * 5, [False, False, False, True, True]]),
            reference_points=torch.rand(B, Q, 4, generator=g) * 0.5 + 0.2, spatial_shapes=shapes,
            level_start_index=lsi, valid_ratios=torch.ones(B, 4, 2), self_attn_mask=None, output_attentions=False,
            output_hidden_states=False, return_dict=True)
    return rec, {"keys": json.dumps([list(k) for k in key_shapes(dec)]), "seed": seed, "config": config_json(cfg)}


def main():
    cfgm, gd = ref_shim.load_gdino()
    np.savez(os.path.join(HERE, "gdino_neck_cpu.npz"), **neck_golden(cfgm, gd))
    rec, extra = dropin_encoder(cfgm, gd)
    rec.save(os.path.join(HERE, "gdino_dropin_enc.npz"), **extra)
    rec, extra = dropin_decoder(cfgm, gd)
    rec.save(os.path.join(HERE, "gdino_dropin_dec.npz"), **extra)
    np.savez(os.path.join(HERE, "gdino_stage_cpu.npz"), **stage_goldens(cfgm, gd))
    np.savez(os.path.join(HERE, "gdino_internimage_cpu.npz"), **internimage_goldens())
    for f in ("gdino_stage_cpu.npz", "gdino_internimage_cpu.npz", "gdino_neck_cpu.npz", "gdino_dropin_enc.npz",
              "gdino_dropin_dec.npz"):
        print(f, os.path.getsize(os.path.join(HERE, f)))


if __name__ == "__main__":
    main()
