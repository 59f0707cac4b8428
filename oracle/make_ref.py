"""Recipe: stage the UNMODIFIED reference under oracle/_ref/ so that it travels with the working tree.

TEST / MEASUREMENT INFRASTRUCTURE (see oracle/__init__.py).  The reference (thinclab/IA2C) has no
setup.py / pyproject.toml — it is nine loose files — so ``pip install --target oracle/_ref <reference>``
has nothing to install.  This recipe is the equivalent: a byte-for-byte copy of the reference's Python
files into ``oracle/_ref/`` (git-ignored: no reference source enters the repository) plus a manifest of
their SHA-256 digests, so that anything that later runs them can prove they are unmodified.

    IA2C_REFERENCE=/path/to/IA2C python -m oracle.make_ref

``__graft_entry__.build()`` runs it whenever the reference checkout (REF_SRC) is present.  Users of the copy:
  * ``bench.py --impl reference`` and bench.py's ``cpu_baseline`` leg — time the reference's own
    ia2c.py loop (oracle/ref_runner.py) on the GPU box's host cores;
  * ``tests/test_gpu_reference_scripts.py`` — execute the unmodified ia2c.py / a2c_org_test.py against
    the drop-in modules on the GPU.
Nothing here is imported by the product package, and no reference source enters git history.
"""
from __future__ import annotations

import hashlib
import json
import os
import shutil

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SRC = os.environ.get("IA2C_REFERENCE", "/root/reference")
REF_DST = os.path.join(ROOT, "oracle", "_ref")
FILES = ("Org.py", "ac_nets.py", "belief_filter_deprecated.py", "ia2c.py", "a2c_org_test.py", "a2c_test.py")
MANIFEST = "MANIFEST.json"


def sha256(path):
    return hashlib.sha256(open(path, "rb").read()).hexdigest()


def stage(src=REF_SRC, dst=REF_DST):
    """Copy the reference files; returns the manifest dict.  Raises if the source tree is absent."""
    if not os.path.isdir(src):
        raise FileNotFoundError(f"reference tree {src} not present (set IA2C_REFERENCE to a checkout of thinclab/IA2C)")
    os.makedirs(dst, exist_ok=True)
    manifest = {"source": src, "files": {}}
    for f in FILES:
        shutil.copyfile(os.path.join(src, f), os.path.join(dst, f))
        manifest["files"][f] = sha256(os.path.join(dst, f))
    json.dump(manifest, open(os.path.join(dst, MANIFEST), "w"), indent=1, sort_keys=True)
    return manifest


def verify(dst=REF_DST):
    """-> manifest if every staged file still has its recorded digest, else raises."""
    path = os.path.join(dst, MANIFEST)
    if not os.path.exists(path):
        raise FileNotFoundError(f"{path} missing: stage the reference with `python -m oracle.make_ref`")
    manifest = json.load(open(path))
    for f, digest in manifest["files"].items():
        got = sha256(os.path.join(dst, f))
        if got != digest:
            raise RuntimeError(f"oracle/_ref/{f} was modified after staging (sha256 {got} != {digest})")
    return manifest


if __name__ == "__main__":
    m = stage()
    print(f"staged {len(m['files'])} unmodified reference files from {m['source']} into {REF_DST}")
