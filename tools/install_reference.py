"""Copy the UNMODIFIED reference (its Python sources only: src/, scripts/, models/, utils/, configs/, train.py, test.py,
eval.py -- ~1.5 MB) from /root/reference into baseline/_ref/, which is git-ignored (never part of this repository's
history) but NOT gpurun-ignored, so it travels to the GPU box.  Used there, and only there, as a measured baseline and as
the caller side of the drop-in boundary:
  * bench.py --impl reference        : the reference module's own CPU forward (kind "reference");
  * bench.py gpu_eager_baseline      : the reference module in PyTorch eager on the same GPU.
Nothing in tests/ reads it: the drop-in boundary tests use oracle/reference_layout.py.
Nothing under image-super-resolution_b200/ imports it.      python tools/install_reference.py [src_root] [dst]
"""
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def install(src="/root/reference", dst=None) -> bool:
    dst = dst or os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(src, "src", "models")):
        return False
    os.makedirs(dst, exist_ok=True)
    ign = shutil.ignore_patterns("__pycache__", "*.pyc", "*.pth", "*.pt", "*.png", "*.jpg", "*.zip")
    for d in ("src", "scripts", "models", "utils", "configs"):
        if os.path.isdir(os.path.join(src, d)):
            shutil.copytree(os.path.join(src, d), os.path.join(dst, d), dirs_exist_ok=True, ignore=ign)
    for f in ("train.py", "test.py", "eval.py", "LICENSE"):
        if os.path.isfile(os.path.join(src, f)):
            shutil.copy2(os.path.join(src, f), os.path.join(dst, f))
    with open(os.path.join(dst, "PROVENANCE.txt"), "w") as fh:
        fh.write("Unmodified copy of the Python sources of Nikhil-AI-Labs/Image-Super-Resolution (from /root/reference),\n"
                 "made by tools/install_reference.py for baseline measurements.  Git-ignored: not part of this repository.\n")
    return True


if __name__ == "__main__":
    ok = install(*(sys.argv[1:3]))
    print("installed" if ok else "reference tree not found: nothing installed")
