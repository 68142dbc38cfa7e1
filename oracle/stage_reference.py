#!/usr/bin/env python
"""Stage the UNMODIFIED reference sources of the hot path under oracle/_ref/ (git-ignored build output, like the
built .so).

    python -m oracle.stage_reference [--src <checkout of kwonminki/Asyrp_official>]

The reference checkout is --src, else $ASYRP_REFERENCE_DIR, else REFERENCE, where the project's reference is mounted
read-only (tests/golden/make_golden.py reads the same one).  Without one there is nothing to stage and the baseline
arms of bench.py use the restatement oracle/ instead.

The reference is a directory of Python scripts without a package, so `pip install --target oracle/_ref` has nothing
to install; this script copies the files `bench.py --impl reference` and the eager-GPU baseline import:
utils/, models/{ddpm,improved_ddpm,guided_diffusion}/, configs/ and the three DeltaBlock checkpoints SURVEY §8(d)
names.  Nothing under oracle/_ref/ is tracked by git or imported by the product package."""
import argparse
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DST = os.path.join(ROOT, "oracle", "_ref")
REFERENCE = "/root/reference"
CKPTS = ["smiling_LC_CelebA_HQ_t999_ninv40_ngen40_0.pth", "dog_happy_LC_dog_t999_ninv40_ngen40_0.pth",
         "church_gothic_LC_church_outdoor_t999_ninv40_ngen40_0.pth"]


def reference_dir():
    """the reference checkout: $ASYRP_REFERENCE_DIR when set, else REFERENCE"""
    return os.environ.get("ASYRP_REFERENCE_DIR") or REFERENCE


def stage(src=None, dst=DST, quiet=False):
    """copy the reference checkout `src` (default: reference_dir()) into `dst`; False when there is none"""
    src = src or reference_dir()
    if not os.path.isdir(src):
        return False
    ig = shutil.ignore_patterns("__pycache__", "*.pyc", "insight_face", "*.tsv")
    for sub in ("utils", "models", "configs"):
        d = os.path.join(dst, sub)
        if os.path.isdir(d):
            shutil.rmtree(d)
        shutil.copytree(os.path.join(src, sub), d, ignore=ig)
    os.makedirs(os.path.join(dst, "checkpoint"), exist_ok=True)
    for c in CKPTS:
        shutil.copy2(os.path.join(src, "checkpoint", c), os.path.join(dst, "checkpoint", c))
    if not quiet:
        n = sum(len(f) for _, _, f in os.walk(dst))
        print(f"staged {n} files from {src} into {dst}")
    return True


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--src", default=None, help="reference checkout (default: $ASYRP_REFERENCE_DIR, else REFERENCE)")
    a = ap.parse_args()
    sys.exit(0 if stage(a.src) else 1)
