"""CPU tests of the "denoise_checkpoints" job key (pathed_b200/host/job.cpp): its default, the values Job refuses, its need of
"denoise": true, and what job_describe reports."""
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


def test_denoise_checkpoints_key_default_and_values(tmp_path):
    assert job_describe(_job(tmp_path))["denoise_checkpoints"] is False
    assert job_describe(_job(tmp_path, denoise=True))["denoise_checkpoints"] is False
    assert job_describe(_job(tmp_path, denoise=True, denoise_checkpoints=None))["denoise_checkpoints"] is False  # null: absent
    assert job_describe(_job(tmp_path, denoise=True, denoise_checkpoints=False))["denoise_checkpoints"] is False
    d = job_describe(_job(tmp_path, denoise=True, denoise_checkpoints=True))
    assert d["denoise_checkpoints"] is True and d["denoise"] is True
    d = job_describe(_job(tmp_path, denoise=True, denoise_checkpoints=True, adaptive_threshold=0.1))
    assert d["denoise_checkpoints"] is True and d["adaptive"] is True
    assert job_describe(_job(tmp_path, denoise_checkpoints=False))["denoise_checkpoints"] is False  # off needs no denoise


@pytest.mark.parametrize("bad", [1, 0, 1.5, "true", [True], {"on": True}])
def test_non_bool_denoise_checkpoints_values_are_refused(tmp_path, bad):
    with pytest.raises(PathedError, match="denoise_checkpoints must be true or false"):
        job_describe(_job(tmp_path, denoise=True, denoise_checkpoints=bad))


@pytest.mark.parametrize("denoise", [None, False])
def test_denoise_checkpoints_need_denoise(tmp_path, denoise):
    over = {} if denoise is None else {"denoise": denoise}
    with pytest.raises(PathedError, match="denoise_checkpoints needs"):
        job_describe(_job(tmp_path, denoise_checkpoints=True, **over))
