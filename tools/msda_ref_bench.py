"""The reference's own MSDA CUDA kernel (oracle/_ref/msda, built by oracle/build_msda_ref.py from the reference's
sources, recompiled for sm_100) timed beside ours on the same B200 at the BASELINE cfg 2b shapes, plus a
GPU-side parity check against it (SURVEY 8c row 2: "the kernel to beat").

    python tools/msda_ref_bench.py [--out profiles/r2_msda_vs_reference_kernel.json]
"""
import argparse
import importlib.util
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def load_reference_ext():
    import torch  # noqa: F401  (libtorch must be loaded first)
    path = os.path.join(ROOT, "oracle", "_ref", "msda", "MultiScaleDeformableAttention.so")
    if not os.path.exists(path):
        return None
    spec = importlib.util.spec_from_file_location("MultiScaleDeformableAttention", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def time_ms(torch, fn, reps=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    tot = 0.0
    for _ in range(reps):
        flush.zero_()                                     # L2 flush between timed launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    return tot / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import bench_workloads as B
    import visionllm_b200.msda as ours
    ref = load_reference_ext()
    dev = torch.device("cuda", 0)
    peaks = B.measured_peaks()
    res = {"device": torch.cuda.get_device_name(0), "hbm_peak_gbs": peaks["hbm_gbs"], "peak_source": peaks["source"],
           "reference_kernel": "visionllmv2/model/unipose/ops/src/cuda/ms_deform_im2col_cuda.cuh "
                               "(ms_deformable_im2col_gpu_kernel), recompiled for sm_100" if ref else "NOT BUILT",
           "cases": {}}
    N = 8
    value, shapes, lsi, loc, attw = B.msda_encoder_inputs(torch, N, dev, 1234)
    S = value.shape[1]
    g = torch.Generator(device=dev).manual_seed(5)

    def dec_inputs(Q):
        ctr = torch.rand(N, Q, 1, 1, 1, 2, device=dev, generator=g)
        wh = torch.rand(N, Q, 1, 1, 1, 2, device=dev, generator=g) * 0.45 + 0.05
        off = torch.randn(N, Q, 8, 4, 4, 2, device=dev, generator=g) * 0.25
        l = (ctr + off * wh * 0.5).contiguous()
        w = torch.softmax(torch.randn(N, Q, 8, 16, device=dev, generator=g), -1).view(N, Q, 8, 4, 4).contiguous()
        return l, w

    cases = {"enc_Lq21760": (loc, attw)}
    for Q in (900, 100):
        cases[f"dec_Lq{Q}"] = dec_inputs(Q)
    for name, (l, w) in cases.items():
        Lq = l.shape[1]
        alg = (value[0].numel() + l[0].numel() + w[0].numel() + Lq * 256) * 4 * N
        row = {"algorithmic_bytes": alg}
        fast = ours.ms_deform_attn_forward(value, shapes, lsi, l, w, 64)
        strict = ours.ms_deform_attn_forward(value, shapes, lsi, l, w, 64, flags=ours.STRICT)
        t = time_ms(torch, lambda: ours.ms_deform_attn_forward(value, shapes, lsi, l, w, 64))
        row["ours_fast"] = {"ms": t, "GBps": alg / t / 1e6, "frac_of_hbm_peak": alg / t / 1e6 / peaks["hbm_gbs"]}
        t = time_ms(torch, lambda: ours.ms_deform_attn_forward(value, shapes, lsi, l, w, 64, flags=ours.STRICT), reps=5)
        row["ours_strict"] = {"ms": t, "GBps": alg / t / 1e6}
        if ref is not None:
            r = ref.ms_deform_attn_forward(value, shapes, lsi, l, w, 64)
            t = time_ms(torch, lambda: ref.ms_deform_attn_forward(value, shapes, lsi, l, w, 64), reps=5)
            row["reference_kernel"] = {"ms": t, "GBps": alg / t / 1e6, "frac_of_hbm_peak": alg / t / 1e6 / peaks["hbm_gbs"]}
            row["speedup_fast_vs_reference_kernel"] = t / row["ours_fast"]["ms"]
            scale = float(r.abs().max())
            row["parity_vs_reference_kernel"] = {
                "fast_max_abs_err": float((fast - r).abs().max()), "strict_max_abs_err": float((strict - r).abs().max()),
                "ref_max_abs": scale,
                # the reference kernel is compiled with nvcc's default -fmad=true, ours strict has no contraction
                # (it follows the CPU-visible arithmetic of the oracle): identical indices, values within fp32 rounding
                "strict_bitwise_equal_fraction": float((strict.view(torch.int32) == r.view(torch.int32)).float().mean()),
            }
        res["cases"][name] = row
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        with open(os.path.join(ROOT, args.out), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
