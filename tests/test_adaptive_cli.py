"""CPU tier: `drt_raytrace --adaptive` refuses several GPUs before it touches a device, so the refusal holds where no GPU exists."""
import os
import subprocess

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(REPO, "daily-ray-trace_b200", "drt_raytrace")


def test_adaptive_refuses_several_gpus(tmp_path):
    if not os.path.exists(BIN):
        pytest.fail("drt_raytrace is not built (make -C daily-ray-trace_b200)")
    run = subprocess.run([BIN, "--adaptive", "0.02", "--gpus", "2"], cwd=str(tmp_path), capture_output=True, text=True, timeout=60)
    assert run.returncode != 0
    assert "--adaptive renders on one GPU" in run.stderr, run.stderr
