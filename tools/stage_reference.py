#!/usr/bin/env python
"""Stage an unmodified checkout of the upstream torch-optical-flow project into `oracle/_ref/reference/`.

The live-model overlay tests (tests/test_reference_overlay.py) and the golden-vector generator
(tests/golden/make_golden.py) need the reference's own `optical_flow` package, `methods/raft/model` and
`tests/operator`, which this repository does not contain.  `__graft_entry__.build()` calls stage() when
OFB200_REFERENCE names a checkout: the three trees are copied byte for byte, nothing edited, into the git-ignored
`oracle/_ref/reference/`, so a copy of the working tree carries them to a machine where the variable is not set.
"""
import hashlib
import json
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DST = os.path.join(ROOT, "oracle", "_ref", "reference")
TREES = ("optical_flow", os.path.join("methods", "raft", "model"), os.path.join("tests", "operator"))


def is_reference(path) -> bool:
    return bool(path) and os.path.isfile(os.path.join(path, "methods", "raft", "model", "raft.py"))


def find_reference():
    """OFB200_REFERENCE when it names a checkout, else a checkout staged under oracle/_ref/, else None."""
    env = os.environ.get("OFB200_REFERENCE")
    if is_reference(env):
        return env
    base = os.path.dirname(DST)
    subdirs = sorted(os.path.join(base, d) for d in os.listdir(base)) if os.path.isdir(base) else []
    return next((p for p in [base] + subdirs if is_reference(p)), None)


def stage(src=None, dst: str = DST) -> bool:
    src = src or os.environ.get("OFB200_REFERENCE")
    if not is_reference(src) or os.path.realpath(src) == os.path.realpath(dst):
        return False
    manifest = {}
    for tree in TREES:
        s, d = os.path.join(src, tree), os.path.join(dst, tree)
        if os.path.isdir(d):
            shutil.rmtree(d)
        shutil.copytree(s, d, ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
        for base, _, files in os.walk(d):
            for f in sorted(files):
                p = os.path.join(base, f)
                manifest[os.path.relpath(p, dst)] = hashlib.sha256(open(p, "rb").read()).hexdigest()
    with open(os.path.join(dst, "MANIFEST.json"), "w") as fh:
        json.dump({"files": manifest}, fh, indent=1, sort_keys=True)
    return True


if __name__ == "__main__":
    ok = stage()
    print(f"staged into {DST}" if ok else "OFB200_REFERENCE does not name a reference checkout: nothing staged")
    sys.exit(0)
