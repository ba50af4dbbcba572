"""bench.py --dump-outputs: what the timed network holds after its last step, as float64 .npy files — identical from run to
run with the same arguments, bounded in size, and (GPU) the same arrays from the device arm as from the oracle arm over
the same window."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, *args):
    out = subprocess.run([sys.executable, "bench.py", "--steps", "4", "--warmup", "1", "--nodes", "1024", "--cpu-max-nodes", "1024",
                          "--dump-outputs", str(out_dir), *args], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-1000:] + out.stderr[-2000:]
    names = sorted(os.listdir(out_dir))
    assert names and all(n.endswith(".npy") for n in names)
    assert sum(os.path.getsize(os.path.join(out_dir, n)) for n in names) <= 64 << 20
    arrays = {n[:-4]: np.load(os.path.join(out_dir, n)) for n in names}
    assert all(a.dtype == np.float64 for a in arrays.values())
    return arrays


def test_reference_arm_dump_is_deterministic_and_follows_steps(tmp_path):
    a = _bench(tmp_path / "a", "--impl", "reference")
    b = _bench(tmp_path / "b", "--impl", "reference")
    assert a.keys() == b.keys() and {"counters", "scalar_card", "verified_sample"} <= a.keys()
    assert all((a[k] == b[k]).all() for k in a)
    assert a["counters"].shape == (5, 1024)
    c = _bench(tmp_path / "c", "--impl", "reference", "--steps", "8")
    assert not (a["counters"] == c["counters"]).all()


@pytest.mark.gpu
def test_device_arm_dump_equals_oracle_arm_on_the_same_window(tmp_path):
    dev = _bench(tmp_path / "dev", "--step-ms", "20", "--no-cpu", "--no-profile")
    ref = _bench(tmp_path / "ref", "--impl", "reference", "--ref-step-ms", "20")
    assert dev.keys() == ref.keys()
    bad = [k for k in dev if dev[k].shape != ref[k].shape or not (dev[k] == ref[k]).all()]
    assert not bad, bad
