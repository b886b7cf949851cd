"""Import the UNMODIFIED reference on CPU: from the checkout of the original project named by DCLL_REFERENCE_ROOT or by
BASELINE.json's reference_path, else from its vendored copy oracle/_ref/ (written by oracle/make_ref.py; git-ignored).

TEST / BASELINE INFRASTRUCTURE.  Used by ``tests/golden/make_golden.py`` (fixture generation),
``tests/test_oracle_vs_reference.py`` (skipped when no reference is present) and by ``bench.py``'s reference arm and
``cpu_baseline`` leg, which time the reference classes themselves on the host cores.  Nothing in the product package
imports this module.

Four shims, none touching arithmetic (SURVEY.md section 8c):
  1. ``apex`` is not installed; the reference imports ``apex.amp`` but every use
     is commented out (dcll/pytorch_libdcll.py:23,705-710).
  2. ``yaml.load`` without a Loader fails on PyYAML >= 6 (networks/__init__.py:11).
  3. ``device = 'cuda'`` module global (dcll/pytorch_libdcll.py:34, imported by
     value at networks/__init__.py:7) is pointed at the CPU.
  4. the layer constructors ``print`` their configuration; silenced.
"""
import contextlib
import io
import os
import sys
import types

from .make_ref import DST as VENDORED_ROOT, is_reference, source_candidates


def _pick_root():
    cands = source_candidates()
    for cand in cands + [VENDORED_ROOT]:
        if is_reference(cand):
            return cand
    return cands[0] if cands else VENDORED_ROOT


REFERENCE_ROOT = _pick_root()


def reference_available():
    return is_reference(REFERENCE_ROOT)


def _check_manifest(root):
    """The vendored copy must be byte-identical to what make_ref.py copied (sha256 manifest)."""
    import hashlib
    import json
    mf = os.path.join(root, "MANIFEST.json")
    if not os.path.isfile(mf):
        return
    for rel, want in json.load(open(mf))["sha256"].items():
        with open(os.path.join(root, rel), "rb") as f:
            got = hashlib.sha256(f.read()).hexdigest()
        if got != want:
            raise RuntimeError("oracle/_ref/%s was modified after vendoring (sha256 mismatch): rerun oracle/make_ref.py" % rel)


_cached = None


def load_reference():
    """Returns (libdcll_module, networks_module, data_utils_module)."""
    global _cached
    if _cached is not None:
        return _cached
    if not reference_available():
        raise RuntimeError("reference not present at %s" % REFERENCE_ROOT)
    _check_manifest(REFERENCE_ROOT)
    if "apex" not in sys.modules:
        apex = types.ModuleType("apex")
        apex.amp = types.ModuleType("apex.amp")
        sys.modules["apex"] = apex
        sys.modules["apex.amp"] = apex.amp
    import yaml

    if not getattr(yaml.load, "_dcll_shim", False):
        _orig = yaml.load

        def _load(stream, Loader=yaml.SafeLoader):
            return _orig(stream, Loader=Loader)

        _load._dcll_shim = True
        yaml.load = _load
    # The reference's top-level package names (dcll, networks, data) are generic;
    # import them under a private path entry and keep them out of the way of the
    # product package, which uses the same sub-module names under its own root.
    sys.path.insert(0, REFERENCE_ROOT)
    try:
        import importlib

        L = importlib.import_module("dcll.pytorch_libdcll")
        L.device = "cpu"
        N = importlib.import_module("networks")
        N.device = "cpu"
        U = importlib.import_module("data.utils")
    finally:
        sys.path.remove(REFERENCE_ROOT)
    _cached = (L, N, U)
    return _cached


@contextlib.contextmanager
def quiet():
    with contextlib.redirect_stdout(io.StringIO()):
        yield


def build_reference_net(spec_name, im_dims, batch_size, target_size, *, arp=0.0, alpha=0.92,
                        alphas=0.85, alpharp=0.65, lc_ampl=0.5, random_tau=True, netscale=1.0,
                        burnin=50, lr=1e-6, beta=0.95, train=True, seed=1):
    """ConvNetwork built exactly as train.py:98-194 does (test_radio_ml.py:92-110 when train=False)."""
    import numpy as np
    import torch

    L, N, _ = load_reference()
    args = types.SimpleNamespace(netscale=netscale, alpha=alpha, alphas=alphas, alpharp=alpharp,
                                 arp=arp, lc_ampl=lc_ampl, random_tau=random_tau)
    torch.manual_seed(seed)
    np.random.seed(seed)
    with quiet():
        convs = N.load_network_spec(os.path.join(REFERENCE_ROOT, "networks", spec_name + ".yaml"))
        if train:
            net = N.ConvNetwork(args, im_dims, batch_size, convs, target_size,
                                act=torch.nn.Sigmoid(), loss=torch.nn.SmoothL1Loss,
                                opt=torch.optim.Adam,
                                opt_param={"betas": [0.0, beta], "weight_decay": 10.0},
                                learning_rates=[lr], burnin=burnin)
        else:
            net = N.ConvNetwork(args, im_dims, batch_size, convs, target_size,
                                act=torch.nn.Sigmoid(), loss=None, opt=None, opt_param={},
                                learning_rates=None, burnin=burnin)
        net.reset(True)
    return net
