"""CPU: the instruction footprint of the bs = 1 GEMV kernel, read from the built library with scripts/sass_footprint.py.

Every decode launch of a layer starts on this kernel's straight-line code, and its instructions compete with the other
warps of the SM for the instruction caches.  The checks keep the image from growing back: one inlined copy of the digit
split, no spills, and a kernel body well under the size it had before the staging and producer loops were rolled.
"""
import importlib.util
import os
import shutil

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "llama2-accessory_b200", "libb200decode.so")


def _footprint():
    spec = importlib.util.spec_from_file_location("sass_footprint", os.path.join(ROOT, "scripts", "sass_footprint.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.skipif(not (shutil.which("nvdisasm") or os.path.isfile("/usr/local/cuda/bin/nvdisasm")),
                    reason="needs the CUDA toolkit's nvdisasm")
def test_gemv1_kernel_footprint():
    from llama2_accessory_b200._build import build
    build()
    kernels = {k["name"]: k for k in _footprint().analyse(LIB)}
    assert set(kernels) == {"void b200::gemv1_kernel<false>(b200::GemvParams)",
                            "void b200::gemv1_kernel<true>(b200::GemvParams)"}
    for name, k in kernels.items():
        assert k["split_copies"] == 1, (name, k["split_copies"])
        assert k["stack"] == 0, (name, k["stack"])
        assert k["body"] < 4000, (name, k["body"])  # 7004 / 7182 before
