"""Golden vectors of the REFERENCE's own MSDA CUDA kernel (oracle/build_msda_ref.py, recompiled for sm_100) for
tests/test_msda_gpu.py::test_forward_matches_the_reference_cuda_kernel.  Needs a GPU and oracle/_ref/msda built.

For each case the inputs are regenerated from the test's own seeds (make_case(seed=21), grad_output from
default_rng(22)); the file records a checksum of them, the full-array max |x| of every result (the tests' tolerance
scale) and a fixed, seeded sample (sample_index) of each result.

    python tests/golden/gen_golden_msda_cuda.py [OUT.npz]
"""
import importlib.util
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    from test_msda_gpu import REF_CUDA_CASES, grad_output, make_case, sample_index
    path = os.path.join(ROOT, "oracle", "_ref", "msda", "MultiScaleDeformableAttention.so")
    spec = importlib.util.spec_from_file_location("MultiScaleDeformableAttention", path)
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    out = {}
    for ci, case in enumerate(REF_CUDA_CASES):
        value, shapes, lsi, loc, attw = make_case(*case, seed=21)
        out[f"c{ci}_checksum"] = np.array([float(a.astype(np.float64).sum()) for a in (value, loc, attw)])
        v, sh, ls, lo, w = (torch.from_numpy(a).cuda() for a in (value, shapes, lsi, loc, attw))
        res = {"out32": ref.ms_deform_attn_forward(v, sh, ls, lo, w, 64)}
        v64, lo64, w64 = v.double(), lo.double(), w.double()
        res["out64"] = ref.ms_deform_attn_forward(v64, sh, ls, lo64, w64, 64)
        go = torch.from_numpy(grad_output(res["out64"].shape)).cuda()
        res["gv"], res["gl"], res["gw"] = ref.ms_deform_attn_backward(v64, sh, ls, lo64, w64, go, 64)
        for k, t in res.items():
            a = t.cpu().numpy().reshape(-1)
            out[f"c{ci}_{k}_absmax"] = np.array(np.abs(a).max())
            out[f"c{ci}_{k}"] = a[sample_index(a.size, ci)]
    dst = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "msda_cuda_ref.npz")
    os.makedirs(os.path.dirname(os.path.abspath(dst)), exist_ok=True)
    np.savez(dst, **out)
    print("wrote", dst, os.path.getsize(dst), "bytes")


if __name__ == "__main__":
    main()
