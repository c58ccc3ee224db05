"""CPU: the drop-in claim of INTEGRATION.md section 4 -- the B200 layer classes can stand in for the reference's under
the REFERENCE'S OWN `GroundingDinoEncoder` / `GroundingDinoDecoder` stacks (their python loops, reference points,
hidden-state bookkeeping).  tests/golden/gen_golden_gdino_cpu.py ran those stacks and recorded every call they made to
their layers and heads (keyword arguments and outputs); here the B200 classes, built under the same parameter names with
the same weights, receive exactly those calls and must return the same outputs.  Kernels are replaced by fp32 torch
stand-ins here (no GPU in this test); the -m gpu tests cover the kernels."""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
from test_gdino_logic_cpu import torch_kernels  # noqa: E402,F401  (fixture)
from test_gdino_model_cpu import reference_config  # noqa: E402


def replay(g, modules, tol):
    """Call modules[name] with every recorded call of the reference module `name`; compare the primary output
    (encoder layer: (vision, text); decoder layer: hidden states; heads: the tensor) within tol[name]."""
    def load(e):
        if "tensor" in e:
            return torch.from_numpy(g[e["tensor"]])
        if "seq" in e:
            return tuple(load(x) for x in e["seq"])
        return e["value"]

    def tensors(x):
        return [x] if isinstance(x, torch.Tensor) else [t for y in x for t in tensors(y)]

    calls = json.loads(str(g["calls"]))
    assert {c["module"] for c in calls} == set(modules)
    for c in calls:
        name = c["module"]
        with torch.no_grad():
            got = modules[name](*[load(a) for a in c["args"]], **{k: load(v) for k, v in c["kwargs"].items()})
        want = load(c["output"])
        if not name.startswith(("bbox_embed", "reference_points_head")):
            got, want = got[0], want[0]
        got, want = tensors(got), tensors(want)
        assert len(got) == len(want), name
        for a, b in zip(got, want):
            assert a.shape == b.shape and (a - b).abs().max() < tol(name), name


def load_weights(stack, g):
    from weights_util import key_shapes, seeded_state_dict
    assert [list(k) for k in key_shapes(stack)] == json.loads(str(g["keys"]))    # identical parameter names
    stack.load_state_dict(seeded_state_dict(stack, int(g["seed"])), strict=True)


def test_reference_encoder_stack_runs_on_b200_layers(golden_dir, torch_kernels):  # noqa: F811
    import visionllm_b200.gdino as b200
    g = np.load(os.path.join(golden_dir, "gdino_dropin_enc.npz"))
    cfg = reference_config(str(g["config"]))
    stack = torch.nn.Module()
    stack.layers = torch.nn.ModuleList([b200.GroundingDinoEncoderLayer(cfg) for _ in range(cfg.encoder_layers)])
    load_weights(stack, g)
    stack.eval()
    replay(g, {f"layers.{i}": layer for i, layer in enumerate(stack.layers)}, lambda name: 1e-4)


def test_reference_decoder_stack_runs_on_b200_layers(golden_dir, torch_kernels):  # noqa: F811
    """The reference's GroundingDinoDecoder (sine box embeddings, query_pos MLP, per-layer box refinement through
    bbox_embed, intermediate stacking) driving B200 decoder layers and B200 MLP heads."""
    import visionllm_b200.gdino_heads as b200h
    from visionllm_b200.gdino_model import _Decoder
    g = np.load(os.path.join(golden_dir, "gdino_dropin_dec.npz"))
    cfg = reference_config(str(g["config"]))
    dec = _Decoder(cfg)
    dec.bbox_embed = torch.nn.ModuleList([b200h.GroundingDinoMLPPredictionHead(256, 256, 4, 3)
                                          for _ in range(cfg.decoder_layers)])
    load_weights(dec, g)
    dec.eval()
    modules = {"reference_points_head": dec.reference_points_head}
    for i in range(cfg.decoder_layers):
        modules[f"layers.{i}"], modules[f"bbox_embed.{i}"] = dec.layers[i], dec.bbox_embed[i]
    replay(g, modules, lambda name: 1e-5 if name.startswith("bbox_embed") else 1e-4)
