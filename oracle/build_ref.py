"""oracle/build_ref.py -- vendors the UNMODIFIED reference into oracle/_ref/ (test / benchmark infrastructure only).

The reference is pure Python, so "building" it is a verbatim copy of the files the hot path needs (model/, core/, config/ of
Janspiry/Image-Super-Resolution-via-Iterative-Refinement) from /root/reference.  oracle/_ref/ is git-ignored (no reference source
enters the history) but NOT gpurun-ignored, so the copy travels to the GPU box, where `bench.py --impl reference` and the
`cpu_baseline` leg import model.networks.define_G from it and time the reference's own p_sample on the host cores.

Nothing on the product path (sr3_b200/, libsr3_b200.so) imports or reads oracle/_ref.

    python oracle/build_ref.py            # no-op (exit 0) when /root/reference is absent, e.g. on the GPU box
"""
import hashlib
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.environ.get("SR3_REFERENCE_ROOT", "/root/reference")
DST = os.path.join(HERE, "_ref")
PARTS = ("model", "core", "config")


def _make_writable(path):
    for root, _dirs, names in os.walk(path):
        os.chmod(root, os.stat(root).st_mode | 0o700)
        for n in names:
            p = os.path.join(root, n)
            os.chmod(p, os.stat(p).st_mode | 0o600)


def build(verbose=True):
    if not os.path.isdir(os.path.join(SRC, "model")):
        if verbose:
            print(f"oracle/build_ref.py: {SRC} not present, keeping whatever is in {DST}")
        return os.path.isdir(os.path.join(DST, "model"))
    manifest = {}
    for part in PARTS:
        s, d = os.path.join(SRC, part), os.path.join(DST, part)
        if not os.path.isdir(s):
            continue
        if os.path.isdir(d):
            _make_writable(d)
            shutil.rmtree(d)
        shutil.copytree(s, d, ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
        _make_writable(d)                      # a read-only source keeps its modes in the copy; the next build must be able to replace it
        for root, _dirs, names in os.walk(d):
            for n in sorted(names):
                p = os.path.join(root, n)
                manifest[os.path.relpath(p, DST)] = hashlib.sha256(open(p, "rb").read()).hexdigest()
    with open(os.path.join(DST, "MANIFEST.json"), "w") as fh:
        json.dump({"source": SRC, "files": manifest}, fh, indent=1, sort_keys=True)
    if verbose:
        print(f"oracle/build_ref.py: copied {len(manifest)} files of the reference into {DST}")
    return True


if __name__ == "__main__":
    sys.exit(0 if build() or True else 1)
