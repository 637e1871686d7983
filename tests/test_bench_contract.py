"""bench.py contract checks: the reference arm runs on the host cores and prints one JSON line with the keys a caller
parses; the GPU arm refuses to run without CUDA (no CPU fallback) and, on a GPU, writes the outputs of its last timed
step when asked to."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          timeout=600, env=e)


def test_reference_arm_json_line():
    r = _run("--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "pairs/s" and line["higher_is_better"] is True
    assert line["metric"].startswith("image-text pairs/sec") and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert "sample" in line["cpu_baseline"] and line["config"]["workload"].startswith("dual tower")
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["gpu_launches"] == 0 and line["steps"] == 1


def test_reference_arm_other_ranks_exit_quietly():
    r = _run("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1",
             env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_gpu_arm_needs_cuda():
    r = _run("--gpus", "1", "--steps", "1", "--warmup", "3")
    assert r.returncode != 0
    assert "no CPU fallback" in r.stdout


def test_bad_arguments_are_refused():
    for args in (("--steps", "0"), ("--impl", "reference", "--dump-outputs", "out"),
                 ("--config", "pairs,cfg3", "--dump-outputs", "out")):
        r = _run(*args)
        assert r.returncode == 2 and "error:" in r.stderr, args


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path, state_dict):
    r = _run("--gpus", "1", "--steps", "2", "--warmup", "3", "--quick", "--no-cpu-baseline", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    assert sorted(os.listdir(tmp_path)) == ["logits_per_image.npy"]
    got = np.load(tmp_path / "logits_per_image.npy")
    assert got.dtype == np.float32 and got.shape == (1024, 1024)
    # step i runs input set i % 2 (seeds 1234 + i / 1235 + i): the last of two steps saw set 1
    from plip_b200 import synthetic as synth
    from plip_b200.distributed import ShardedCLIP
    from plip_b200.engine import Engine
    eng = Engine(state_dict, max_micro_batch=1024)
    px = synth.pixel_values(1024, seed=1235).to(torch.bfloat16).cuda()
    ids = synth.token_ids(1024, seed=1236, full_length=True)[0].cuda()
    want = ShardedCLIP.from_engine(eng).clip_forward(px, ids).cpu().numpy()
    eng.close()
    assert np.abs(got - want).max() < 1e-3
