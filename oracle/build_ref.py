"""Build recipe for the reference's own CUDA extensions (TEST INFRASTRUCTURE ONLY).

Compiles the two native extensions of uzh-rpg/dagr *from the sources where they lie*
under /root/reference (nothing is copied into this repo) into oracle/_ref/:

  ev_graph_cuda  <- /root/reference/src/dagr/graph/ev_graph.cu (+ spiral.h)       (setup.py:8-9)
  asy_tools      <- /root/reference/src/dagr/asynchronous/asy_tools/main.cu      (setup.py:10-11)

The products are git-ignored (oracle/_ref/).  tests/golden/make_reference_kernels_golden.py
runs them on a GPU to write the fixtures the `-m gpu` tests compare our kernels against.
Without the reference sources this script builds nothing.
"""
import os
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
OUT = HERE / "_ref"
REF = Path(os.environ.get("DAGR_REFERENCE", "/root/reference"))

TARGETS = {
    "ev_graph_cuda": REF / "src/dagr/graph/ev_graph.cu",
    "asy_tools": REF / "src/dagr/asynchronous/asy_tools/main.cu",
}


def built(name: str) -> bool:
    return any(OUT.glob(f"{name}/{name}*.so")) or any(OUT.glob(f"{name}*.so"))


def build(verbose: bool = False) -> dict:
    status = {}
    OUT.mkdir(exist_ok=True)
    for name, src in TARGETS.items():
        if built(name):
            status[name] = "prebuilt"
            continue
        if not src.exists():
            status[name] = "reference sources absent"
            continue
        os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0a")
        from torch.utils.cpp_extension import load
        bdir = OUT / name
        bdir.mkdir(exist_ok=True)
        load(name=name, sources=[str(src)], build_directory=str(bdir),
             extra_cuda_cflags=["-O2", "-gencode", "arch=compute_100a,code=sm_100a", "-w"],
             extra_cflags=["-O2", "-w"], is_python_module=False, verbose=verbose)
        status[name] = "built"
    return status


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv))
