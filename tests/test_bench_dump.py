"""`bench.py --dump-outputs DIR`: what the timed path returned in its last step, as float .npy files of at most 64 MB, from
seeded inputs, so that two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("alignments", "linear_outputs_frames", "linear_outputs_sampled", "mel_outputs", "steps")


def run_bench(out_dir, steps, *args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "0", *args,
                        "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == steps
    assert sorted(os.listdir(out_dir)) == sorted(n + ".npy" for n in NAMES)
    d = {n: np.load(os.path.join(out_dir, n + ".npy")) for n in NAMES}
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert sum(os.path.getsize(os.path.join(out_dir, n + ".npy")) for n in NAMES) <= 64 * 10**6
    dec_steps = int(d["steps"][0])
    T = dec_steps * bench.R
    assert d["mel_outputs"].shape == (bench.BATCH, T, 80) and d["alignments"].shape == (bench.BATCH, bench.T_IN, dec_steps)
    frames = d["linear_outputs_frames"]
    assert d["linear_outputs_sampled"].shape == (bench.BATCH, len(frames), 1025)
    assert len(frames) == min(bench.DUMP_LINEAR_FRAMES, T) and np.all(np.diff(frames) > 0) and frames[-1] < T
    return d


def test_reference_arm_dump(tmp_path):
    d = run_bench(tmp_path / "dump", 1, "--impl", "reference")
    assert np.isfinite(d["mel_outputs"]).all() and np.isfinite(d["linear_outputs_sampled"]).all()


@pytest.mark.gpu
def test_gpu_arm_dump_is_what_the_path_returns(tmp_path):
    """The dump of the timed path equals a plain forward of the same seeded batch (rank 0's first batch, weights seed 1234)."""
    import torch
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.hparams import HParams
    from tacotron_multispeaker_b200.weights import random_init
    got = run_bench(tmp_path / "dump", 3, "--inflight", "2", "--e2e-lanes", "2", "--no-cpu", "--no-latency", "--no-vocoder",
                    "--no-throughput-mode", "--no-configs")
    hp = HParams(outputs_per_step=bench.R, max_iters=bench.MAX_ITERS)
    eng = Engine(hp, bench.ID_NUM, 0)
    try:
        eng.load_weights(random_init(hp, bench.ID_NUM, seed=1234))
        want = bench.dump_arrays(*eng.forward(*bench.make_batch(1)))
        torch.cuda.synchronize()
    finally:
        eng.close()
    assert got["steps"][0] == want["steps"][0]
    for name in NAMES:
        np.testing.assert_allclose(got[name], want[name], rtol=0, atol=1e-5, err_msg=name)
