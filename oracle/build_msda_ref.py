"""Build the REFERENCE's own MSDA CUDA extension (the kernel to beat, SURVEY 8c row 2 / BASELINE.md 4b) for sm_100.

Sources are taken where they lie in a VisionLLMv2 checkout (visionllmv2/model/unipose/ops/src -- the same kernels as
mmcv's ms_deform_attn_cuda_kernel.cuh): $VISIONLLMV2_SRC when set, else the first of REFERENCE_CHECKOUTS that exists.
They are copied UNMODIFIED into oracle/_ref/msda/src (git-ignored, never committed), then three mechanical API-compat
edits are applied to the copies so that they compile against torch 2.11:
  * `#include <THC/THCAtomics.cuh>`  -> `#include <ATen/cuda/Atomic.cuh>`   (THC was removed from torch)
  * `x.type().is_cuda()`             -> `x.is_cuda()`
  * `AT_DISPATCH_FLOATING_TYPES(value.type(), ...)` -> `value.scalar_type()`; `.data<T>()` -> `.data_ptr<T>()`
No kernel arithmetic is touched.  Output: oracle/_ref/msda/MultiScaleDeformableAttention.so, loaded by
`tools/msda_ref_bench.py`, bench.py's `msda` object and tests/golden/gen_golden_msda_cuda.py when present.

    python oracle/build_msda_ref.py          (no GPU needed: nvcc cross-compiles; __graft_entry__.build() runs it
                                              when the .so is missing and a reference checkout is found)
"""
import glob
import os
import re
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DST = os.path.join(ROOT, "oracle", "_ref", "msda")
NAME = "MultiScaleDeformableAttention"
SO = os.path.join(DST, NAME + ".so")
OPS_SRC = os.path.join("visionllmv2", "model", "unipose", "ops", "src")
# where the original project's checkout is looked for: next to this repository, and where SURVEY.md's build
# container mounts it
REFERENCE_CHECKOUTS = [os.path.join(os.path.dirname(ROOT), "reference", "VisionLLMv2"), "/root/reference/VisionLLMv2"]


def reference_sources():
    """The reference's MSDA extension sources, or None when no VisionLLMv2 checkout can be read."""
    roots = [os.environ["VISIONLLMV2_SRC"]] if os.environ.get("VISIONLLMV2_SRC") else REFERENCE_CHECKOUTS
    for root in roots:
        path = os.path.join(root, OPS_SRC)
        if os.path.isdir(path) and os.access(path, os.R_OK | os.X_OK):
            return path
    return None


def main():
    ref_src = reference_sources()
    if ref_src is None:
        print("no readable VisionLLMv2 checkout (set VISIONLLMV2_SRC): nothing to build")
        return 1
    src = os.path.join(DST, "src")
    shutil.rmtree(src, ignore_errors=True)
    shutil.copytree(ref_src, src)
    for dirpath, _, files in os.walk(src):                 # the copies keep the checkout's modes, possibly read-only
        os.chmod(dirpath, 0o755)
        for f in files:
            os.chmod(os.path.join(dirpath, f), 0o644)
    for path in glob.glob(os.path.join(src, "**", "*.*"), recursive=True):
        text = open(path).read()
        new = text.replace("#include <THC/THCAtomics.cuh>", "#include <ATen/cuda/Atomic.cuh>")
        new = new.replace(".type().is_cuda()", ".is_cuda()")
        new = re.sub(r"AT_DISPATCH_FLOATING_TYPES\((\w+)\.type\(\)", r"AT_DISPATCH_FLOATING_TYPES(\1.scalar_type()", new)
        new = re.sub(r"\.data<", ".data_ptr<", new)
        if new != text:
            open(path, "w").write(new)
    os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0")
    os.environ.setdefault("MAX_JOBS", "8")
    from torch.utils.cpp_extension import load
    build = os.path.join(DST, "build")
    os.makedirs(build, exist_ok=True)
    load(name=NAME, sources=[os.path.join(src, "vision.cpp"), os.path.join(src, "cpu", "ms_deform_attn_cpu.cpp"),
                             os.path.join(src, "cuda", "ms_deform_attn_cuda.cu")],
         extra_include_paths=[src], extra_cflags=["-DWITH_CUDA", "-O3"],
         extra_cuda_cflags=["-DWITH_CUDA", "-O3", "-lineinfo", "-DCUDA_HAS_FP16=1", "-D__CUDA_NO_HALF_OPERATORS__",
                            "-D__CUDA_NO_HALF_CONVERSIONS__", "-D__CUDA_NO_HALF2_OPERATORS__"],
         build_directory=build, is_python_module=False, verbose=True)
    so = glob.glob(os.path.join(build, NAME + "*.so"))[0]
    shutil.copy(so, SO)
    print("built", SO)
    return 0


if __name__ == "__main__":
    sys.exit(main())
