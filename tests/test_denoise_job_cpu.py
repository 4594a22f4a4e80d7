"""CPU tests of the "denoise" job key (pathed_b200/host/job.cpp): its default, the values Job refuses, and what job_describe reports."""
import json

import pytest

from pathed_b200 import PathedError, job_describe


def _job(tmp_path, **over):
    job = {"spp": 64, "integrator": "PathTracer", "scene": "scenes/cornell.json", "startBounce": 0, "lastBounce": 10,
           "output_directory": str(tmp_path / "out"), "output_name": "final", "showUI": False, "force": True, "width": 32, "height": 24}
    job.update(over)
    path = str(tmp_path / "job.json")
    json.dump(job, open(path, "w"))
    return path


def test_denoise_key_default_and_values(tmp_path):
    assert job_describe(_job(tmp_path))["denoise"] is False
    assert job_describe(_job(tmp_path, denoise=None))["denoise"] is False  # null: the key is absent
    assert job_describe(_job(tmp_path, denoise=False))["denoise"] is False
    assert job_describe(_job(tmp_path, denoise=True))["denoise"] is True
    d = job_describe(_job(tmp_path, denoise=True, adaptive_threshold=0.1))
    assert d["denoise"] is True and d["adaptive"] is True


@pytest.mark.parametrize("bad", [1, 0, 1.5, "true", [True], {"on": True}])
def test_non_bool_denoise_values_are_refused(tmp_path, bad):
    with pytest.raises(PathedError, match="denoise must be true or false"):
        job_describe(_job(tmp_path, denoise=bad))


def test_denoise_needs_two_samples(tmp_path):
    with pytest.raises(PathedError, match="denoise needs spp >= 2"):
        job_describe(_job(tmp_path, denoise=True, spp=1))
    assert job_describe(_job(tmp_path, denoise=True, spp=2))["denoise"] is True
    assert job_describe(_job(tmp_path, denoise=False, spp=1))["spp"] == 1
