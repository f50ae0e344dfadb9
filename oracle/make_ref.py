#!/usr/bin/env python
"""Vendor the UNMODIFIED reference package into oracle/_ref/ (git-ignored).

    python oracle/make_ref.py

The reference is pure Python, so "building" it is a copy of
/root/reference/mdp_playground/ (only envs/ and spaces/ -- the step path; the
analysis / Ray config processor are not needed) to oracle/_ref/mdp_playground/.
oracle/_ref/ is listed in .gitignore (no reference source enters the history)
but NOT in .gpurunignore, so it travels to the GPU box with the snapshot like
the built .so files.  There `bench.py` times the reference's own RLToyEnv loop
on the host cores (`cpu_baseline.kind = "reference"`, `--impl reference`).
gymnasium is not installed in the image: the reference is imported through
oracle/gymnasium_standin (see oracle/ref_loader.py).  A MANIFEST with the
sha256 of every copied file is written next to the copy.
"""
import hashlib
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.environ.get("MDPP_REFERENCE_ROOT", "/root/reference")
DST = os.path.join(HERE, "_ref")
KEEP = ("__init__.py", "envs", "spaces")


def main():
    pkg = os.path.join(SRC, "mdp_playground")
    if not os.path.isdir(pkg):
        print("reference checkout not found at", SRC, "- nothing vendored")
        return 0
    out = os.path.join(DST, "mdp_playground")
    if os.path.isdir(DST):
        shutil.rmtree(DST)
    os.makedirs(out)
    manifest = []
    for name in KEEP:
        s, d = os.path.join(pkg, name), os.path.join(out, name)
        if os.path.isdir(s):
            shutil.copytree(s, d, ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
        else:
            shutil.copy2(s, d)
    # the experiment files tests/test_sweep.py reads (REFERENCE_ROOT/experiments)
    exps = os.path.join(SRC, "experiments")
    if os.path.isdir(exps):
        shutil.copytree(exps, os.path.join(DST, "experiments"),
                        ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
    for root, _, files in os.walk(DST):
        for f in sorted(files):
            p = os.path.join(root, f)
            manifest.append((hashlib.sha256(open(p, "rb").read()).hexdigest(),
                             os.path.relpath(p, DST)))
    with open(os.path.join(DST, "MANIFEST.sha256"), "w") as f:
        for h, p in sorted(manifest, key=lambda x: x[1]):
            f.write(f"{h}  {p}\n")
    print(f"vendored {len(manifest)} files into {DST}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
