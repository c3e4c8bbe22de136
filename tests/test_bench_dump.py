"""bench.py --dump-outputs: the seals of the last timed step are written as exact float64 copies, and they are the seals the
CPU oracle proves from the same seeds (so two builds, or two runs, compare seal for seal)."""
import json
import os
import subprocess
import sys
import numpy as np
import pytest
from conftest import DEFAULT, TRACE_SEED, make_segment

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_bench_dump_outputs_match_the_oracle(orc, tmp_path):
    po2, steps, inflight = 12, 2, 2
    env = {k: v for k, v in os.environ.items() if k != "HFB200_DETERMINISTIC_BLINDING"}  # the flag alone must make the seals reproducible
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--po2", str(po2), "--steps", str(steps), "--warmup", "3",
           "--inflight", str(inflight), "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(tmp_path)]
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-4000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["config"]["inflight_per_gpu"] == inflight
    assert sorted(os.listdir(tmp_path)) == ["seal_rank0_ctx%d.npy" % i for i in range(inflight)]
    for slot in range(inflight):
        got = np.load(tmp_path / ("seal_rank0_ctx%d.npy" % slot))
        assert got.dtype == np.float64
        # the seeds bench.py gives context `slot` of rank 0: its trace, and its blinding in the last timed step
        cir, g, code, data = make_segment(orc, DEFAULT, po2, trace_seed=TRACE_SEED + 7919 * slot, blind_seed=1)
        oseal, _, _ = cir.prove(po2, g, code, data, 1 + 17 * (steps - 1) + 101 * slot)
        assert np.array_equal(got, oseal.astype(np.float64))
