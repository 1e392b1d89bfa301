"""Stages the original example's training script for `bench.py --impl reference`.

The original project is plain Python files, so "building" it means copying the two files the reference arm imports,
unmodified, into ``oracle/_ref/`` (kept out of git).  The checkout to copy from is named by ``VIT_REFERENCE_DIR``;
without it nothing is staged and the reference arm reports itself unavailable.

    VIT_REFERENCE_DIR=<checkout of the original example> python -m oracle.reference
"""
from __future__ import annotations

import os
import shutil

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, "_ref")
FILES = ("run_vit_training.py", "utils.py")


def is_staged() -> bool:
    return all(os.path.isfile(os.path.join(REF_DIR, f)) for f in FILES)


def build() -> str | None:
    """Copy the files from ``$VIT_REFERENCE_DIR`` into ``oracle/_ref/``; returns that directory, or None when the
    variable is unset."""
    src = os.environ.get("VIT_REFERENCE_DIR")
    if not src:
        return None
    missing = [f for f in FILES if not os.path.isfile(os.path.join(src, f))]
    if missing:
        raise FileNotFoundError(f"VIT_REFERENCE_DIR={src} lacks {', '.join(missing)}")
    os.makedirs(REF_DIR, exist_ok=True)
    for f in FILES:
        shutil.copyfile(os.path.join(src, f), os.path.join(REF_DIR, f))
    return REF_DIR


if __name__ == "__main__":
    print(build() or "VIT_REFERENCE_DIR is not set: nothing staged")
