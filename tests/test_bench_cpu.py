"""bench.py host logic that needs no GPU: the CPU arm runs the vendored reference, both arms share one config."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")


@pytest.mark.skipif(not os.path.isfile(os.path.join(REF, "MANIFEST.json")), reason="oracle/_ref not vendored (python oracle/make_ref.py)")
def test_reference_arm_runs_vendored_reference():
    env = dict(os.environ, DCLL_REFERENCE_ROOT=REF)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload",
                        "radio_ml_conv_train_16x16_B64", "--steps", "1", "--warmup", "0", "--timesteps", "64"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["cpu_baseline"]["kind"] == "reference" and line["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["unit"] == "windows/s"
    import bench
    import argparse
    a = argparse.Namespace(workload="radio_ml_conv_train_16x16_B64", timesteps=64)
    assert line["config"] == bench.config_dict(a, 1)          # what the B200 arm prints for the same flags


def test_vendored_reference_manifest_guard(tmp_path):
    """A modified vendored copy is refused (sha256 manifest).  The copy is vendored by make_ref from a stand-in source
    tree: the guard reads the manifest before it imports anything."""
    from oracle.make_ref import FILES, make_ref
    src, dst = tmp_path / "src", tmp_path / "_ref"
    for rel in FILES:
        (src / rel).parent.mkdir(parents=True, exist_ok=True)
        (src / rel).write_text("# %s\n" % rel)
    assert make_ref(str(src), verbose=False, dst=str(dst))
    code = "import os,sys; sys.path.insert(0, %r); os.environ['DCLL_REFERENCE_ROOT']=%r\nfrom oracle import refshim\nrefshim.load_reference()" % (ROOT, str(dst))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    with open(dst / "data" / "utils.py", "a") as f:
        f.write("\n# tampered\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode != 0 and "sha256 mismatch" in r.stderr


def test_global_batch_workload_splits_over_ranks():
    import bench
    assert bench.workload("radio_ml_conv_train_dp_global8192_16x16", 8)[2] == 1024
    assert bench.workload("radio_ml_conv_train_dp_global8192_16x16", 2)[2] == 4096
    assert bench.workload("radio_ml_conv_train_dp_global8192_16x16", 8)[6] == "strong"
    assert bench.workload("radio_ml_conv_train_128x128_B64", 8)[2:3] == (64,) and bench.workload("radio_ml_conv_train_128x128_B64", 8)[6] == "weak"
