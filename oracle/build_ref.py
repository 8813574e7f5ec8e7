"""TEST INFRASTRUCTURE ONLY -- compiles the REFERENCE's own CUDA query extension (two source files, read in place from the
reference tree; nothing is copied) into oracle/_ref/ (git-ignored).  It is the un-modified `query_worldcoords_cuda` torch
extension that the reference's models/neural_points/point_query.py:15-22 JIT-builds at import; oracle/make_ref_kernel_golden.py
runs it on a B200 to record the fixtures tests/golden/ref_kernel_*.npz that pin libpnb200's integer query path.

    python -m oracle.build_ref        # needs the reference tree (oracle/ref_shim.py: REF); nvcc cross-compiles for sm_100a
"""
import os
import sys

from oracle import ref_shim

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SRC = os.path.join(ref_shim.REF, "models", "neural_points", "cuda")
OUT = os.path.join(ROOT, "oracle", "_ref")
NAME = "query_worldcoords_cuda"


def build(verbose=False):
    if not os.path.isdir(REF_SRC):
        raise RuntimeError("oracle.build_ref needs the reference's sources at %s" % REF_SRC)
    os.makedirs(OUT, exist_ok=True)
    os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0a")      # no GPU here: name the target instead of probing one
    from torch.utils.cpp_extension import load
    return load(name=NAME, sources=[os.path.join(REF_SRC, f) for f in ("query_worldcoords.cpp", "query_worldcoords.cu")],
                build_directory=OUT, verbose=verbose, extra_cuda_cflags=["-lineinfo"])


def load_prebuilt():
    """Import the extension built by build() (needs neither a compiler nor the reference tree)."""
    import importlib.util
    import torch  # noqa: F401  (libtorch symbols must be loaded first)
    path = os.path.join(OUT, NAME + ".so")
    if not os.path.isfile(path):
        return None
    spec = importlib.util.spec_from_file_location(NAME, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


if __name__ == "__main__":
    m = build(verbose=True)
    print("built", os.path.join(OUT, NAME + ".so"), "exports", [n for n in dir(m) if not n.startswith("_")])
