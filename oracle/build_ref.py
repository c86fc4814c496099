#!/usr/bin/env python3
"""TEST INFRASTRUCTURE ONLY - builds the *reference's own* CUDA extension as `quant_cuda_ref`.

Recipe for `oracle/_ref/` (git-ignored, travels to the GPU box with gpurun):

  * sources are read where they lie: /root/reference/squeezellm/quant_cuda.cpp and
    /root/reference/squeezellm/quant_cuda_kernel.cu - nothing is copied into this repo;
  * the unmodified `.cu` does not compile against torch 2.11 (SURVEY.md section 8(c)):
    `AT_DISPATCH_FLOATING_TYPES(mat.type(), ...)` at quant_cuda_kernel.cu:261,307,367,421,474,545,
    618,699 needs `mat.scalar_type()`.  The patch is applied by `sed` into a scratch directory
    under /tmp (8 sites, a dtype-dispatch macro argument only; no arithmetic is touched);
  * the module is built under the name `quant_cuda_ref` (TORCH_EXTENSION_NAME) for sm_100 so it
    can live in the same process as our own `quant_cuda`;
  * only the resulting `.so` is written to oracle/_ref/.

The product (squeezellm_b200/, bench.py's own arm) never imports this, nor do the tests.  Users:
tests/golden/make_golden_gpu.py and tests/golden/make_golden_parity.py (the reference outputs the tests compare
against), oracle/ref_gpu_timing.py.
"""
import glob
import os
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("SQLLM_REFERENCE_DIR", "/root/reference")
OUT = os.path.join(HERE, "_ref")

SETUP = r"""
from setuptools import setup
from torch.utils import cpp_extension
setup(
    name="quant_cuda_ref",
    ext_modules=[cpp_extension.CUDAExtension(
        "quant_cuda_ref", ["quant_cuda.cpp", "quant_cuda_kernel.cu"],
        extra_compile_args={"cxx": ["-O2"], "nvcc": ["-O2", "-lineinfo"]})],
    cmdclass={"build_ext": cpp_extension.BuildExtension},
)
"""


def have_ref_so():
    return sorted(glob.glob(os.path.join(OUT, "quant_cuda_ref*.so")))


def build(force=False):
    """Build oracle/_ref/quant_cuda_ref*.so.  Returns the path, or None if the reference tree is absent."""
    so = have_ref_so()
    if so and not force:
        return so[0]
    src = os.path.join(REF, "squeezellm")
    if not os.path.isfile(os.path.join(src, "quant_cuda_kernel.cu")):
        return None  # GPU box: /root/reference does not exist, the prebuilt .so travels instead
    os.makedirs(OUT, exist_ok=True)
    tmp = tempfile.mkdtemp(prefix="sqllm_ref_build_")
    try:
        shutil.copy(os.path.join(src, "quant_cuda.cpp"), os.path.join(tmp, "quant_cuda.cpp"))
        with open(os.path.join(src, "quant_cuda_kernel.cu")) as f:
            cu = f.read()
        n = cu.count("mat.type()")
        assert n == 8, f"expected 8 mat.type() dispatch sites, found {n}"
        cu = cu.replace("mat.type()", "mat.scalar_type()")
        with open(os.path.join(tmp, "quant_cuda_kernel.cu"), "w") as f:
            f.write(cu)
        with open(os.path.join(tmp, "setup.py"), "w") as f:
            f.write(SETUP)
        env = dict(os.environ)
        env["TORCH_CUDA_ARCH_LIST"] = "10.0"
        env.setdefault("MAX_JOBS", "4")
        subprocess.check_call([sys.executable, "setup.py", "build_ext", "--inplace"], cwd=tmp, env=env)
        built = glob.glob(os.path.join(tmp, "quant_cuda_ref*.so"))
        assert built, "reference build produced no .so"
        dst = os.path.join(OUT, os.path.basename(built[0]))
        shutil.copy(built[0], dst)
        return dst
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def load():
    """Import the prebuilt reference module (needs torch; kernels need a GPU)."""
    so = have_ref_so()
    if not so:
        raise ImportError("oracle/_ref/quant_cuda_ref*.so not built (run oracle/build_ref.py where /root/reference exists)")
    import importlib.util
    import torch  # noqa: F401  (libtorch must be loaded first)
    spec = importlib.util.spec_from_file_location("quant_cuda_ref", so[0])
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


if __name__ == "__main__":
    p = build(force="--force" in sys.argv)
    print("oracle/_ref:", p)
