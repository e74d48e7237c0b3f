"""TEST INFRASTRUCTURE ONLY -- stages the reference's own Python model package next to the oracle so that it can travel
to the GPU box (where /root/reference does not exist) and be EXECUTED there, unmodified, on the CUDA operator surface.

    python oracle/stage_ref.py        (also run by __graft_entry__.build() in the build container)

Copies `/root/reference/pretrain/pointcontrast/model/` (res16unet.py, resnet.py, modules/) byte for byte into
`oracle/_ref/pointcontrast/model/`.  `oracle/_ref/` is git-ignored (never part of the history, like the built .so files).
Nothing in the product path imports it; `tests/refload.py` does, for the CPU baseline of `bench.py` (the reference's model
file on the oracle operators).  The reference's arithmetic layer (MinkowskiEngine
0.4.3, C++/CUDA) is not under /root/reference, so there is nothing to compile (DESIGN.md "Oracle").
"""
import os
import shutil

SRC = "/root/reference/pretrain/pointcontrast/model"
DST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref", "pointcontrast", "model")


def stage(verbose=False):
    if not os.path.isdir(SRC):
        return False
    if os.path.isdir(DST):
        shutil.rmtree(DST)
    shutil.copytree(SRC, DST, ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
    if verbose:
        print("staged", SRC, "->", DST)
    return True


if __name__ == "__main__":
    print("staged" if stage(True) else f"{SRC} not present: nothing staged")
