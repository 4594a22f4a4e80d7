"""CPU tests of the adaptive sampling job keys (pathed_b200/host/job.cpp): defaults, what Job refuses, and the one-GPU rule of the
`pathed` command-line renderer, which refuses before it touches a device."""
import json
import os
import subprocess

import pytest

from pathed_b200 import PathedError, job_describe
from pathed_b200._binding import PKG_DIR, REPO_ROOT


def _job(tmp_path, **over):
    job = {"spp": 64, "integrator": "PathTracer", "scene": "scenes/cornell.json", "startBounce": 0, "lastBounce": 10,
           "output_directory": str(tmp_path / "out"), "output_name": "final", "showUI": False, "force": True, "width": 32, "height": 24}
    job.update(over)
    path = str(tmp_path / "job.json")
    json.dump(job, open(path, "w"))
    return path


def test_adaptive_keys_and_defaults(tmp_path):
    d = job_describe(_job(tmp_path))
    assert d["adaptive"] is False and d["spp"] == 64
    d = job_describe(_job(tmp_path, adaptive_threshold=0.05))
    assert d["adaptive"] is True and d["adaptive_threshold"] == pytest.approx(0.05)
    assert (d["adaptive_min_spp"], d["adaptive_step_spp"], d["spp"]) == (16, 16, 64)
    d = job_describe(_job(tmp_path, adaptive_threshold=0.2, adaptive_min_spp=2, adaptive_step_spp=1, spp=2))
    assert (d["adaptive_min_spp"], d["adaptive_step_spp"], d["spp"]) == (2, 1, 2)


@pytest.mark.parametrize("bad", [
    {"adaptive_threshold": 0}, {"adaptive_threshold": -0.1}, {"adaptive_threshold": "0.1"},
    {"adaptive_threshold": 0.1, "adaptive_min_spp": 1}, {"adaptive_threshold": 0.1, "adaptive_step_spp": 0},
    {"adaptive_threshold": 0.1, "adaptive_min_spp": 2.5}, {"adaptive_threshold": 0.1, "adaptive_step_spp": "4"},
    {"adaptive_threshold": 0.1, "adaptive_min_spp": 32, "spp": 16}, {"adaptive_threshold": 0.1, "gpus": 2}])
def test_invalid_adaptive_values_are_refused(tmp_path, bad):
    with pytest.raises(PathedError):
        job_describe(_job(tmp_path, **bad))


def test_cli_refuses_an_adaptive_job_on_two_gpus(tmp_path):
    path = _job(tmp_path, adaptive_threshold=0.1, gpus=2)
    r = subprocess.run([os.path.join(PKG_DIR, "pathed"), path, "--root", REPO_ROOT], capture_output=True, text=True)
    assert r.returncode == 1 and "adaptive sampling runs on one GPU" in r.stdout, r.stdout + r.stderr
    assert not os.path.exists(str(tmp_path / "out"))  # refused before the job's output directory was made
