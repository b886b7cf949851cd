#!/usr/bin/env python
"""Vendors the UNMODIFIED reference sources of the hot path into oracle/_ref/ (TEST / BASELINE INFRASTRUCTURE).

    python oracle/make_ref.py --src <checkout of the original project>

The reference is pure Python over torch, so "building" it is a byte-for-byte copy of the few files the path lives in:

    dcll/__init__.py, dcll/pytorch_libdcll.py      the layers and DCLLClassification      (SURVEY section 8a: a2-a9)
    networks/__init__.py, networks/*.yaml           ConvNetwork, load_network_spec, specs  (a10)
    data/__init__.py, data/utils.py                 iq2spiketrain, to_one_hot              (a1)

The source is the checkout named by DCLL_REFERENCE_ROOT, else the one BASELINE.json names as reference_path.
oracle/_ref/ is git-ignored (reference sources never enter the history): `bench.py --impl reference` and the cpu_baseline
leg import the reference classes from there (oracle/refshim.py: apex stub, yaml Loader default, device = 'cpu' -- none
touches arithmetic) and time THEM on the host cores.  A MANIFEST with sha256 of every file is written next to the copies;
refshim checks it on import, so a modified copy is refused.  Called by __graft_entry__.build(), which vendors the
original project wherever that source holds it.
"""
import hashlib
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, "_ref")
BASELINE = os.path.join(os.path.dirname(HERE), "BASELINE.json")
FILES = ["dcll/__init__.py", "dcll/pytorch_libdcll.py", "networks/__init__.py", "networks/radio_ml_conv.yaml",
         "networks/mnist_conv.yaml", "networks/radio_ml_conv_ref.yaml", "data/__init__.py", "data/utils.py",
         "data/load_radio_ml.py"]


def source_candidates():
    """Checkouts of the original project to look in, in order: DCLL_REFERENCE_ROOT, then BASELINE.json's reference_path."""
    out = [os.environ.get("DCLL_REFERENCE_ROOT")]
    try:
        with open(BASELINE) as f:
            out.append(json.load(f).get("reference_path"))
    except (OSError, ValueError):
        pass
    return [c for c in out if c]


def is_reference(root):
    return os.path.isfile(os.path.join(root, "dcll", "pytorch_libdcll.py"))


def sha256(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        h.update(f.read())
    return h.hexdigest()


def make_ref(src=None, verbose=True, dst=DST):
    if src is None:
        src = next((c for c in source_candidates() if is_reference(c)), None)
    if not src or not is_reference(src) or os.path.realpath(src) == os.path.realpath(dst):
        if verbose:
            print("make_ref: no reference at %s, keeping %s as it is" % (src or " or ".join(source_candidates()) or "-", dst))
        return False
    manifest = {}
    for rel in FILES:
        s, d = os.path.join(src, rel), os.path.join(dst, rel)
        os.makedirs(os.path.dirname(d), exist_ok=True)
        shutil.copyfile(s, d)
        manifest[rel] = sha256(d)
    with open(os.path.join(dst, "MANIFEST.json"), "w") as f:
        json.dump({"source": src, "sha256": manifest}, f, indent=1, sort_keys=True)
    if verbose:
        print("make_ref: %d reference files -> %s" % (len(FILES), dst))
    return True


if __name__ == "__main__":
    src = sys.argv[sys.argv.index("--src") + 1] if "--src" in sys.argv else None
    sys.exit(0 if make_ref(src) else 1)
