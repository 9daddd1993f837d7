"""GPU: bench.py times as many steps as --steps asks for, and --dump-outputs writes what the last timed step returned; the
same inputs give the same outputs whatever the step count."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_steps_are_timed_and_dump_outputs_repeat(cuda, tmp_path):
    lines, dumped = {}, {}
    for steps in (1, 3):
        out = tmp_path / ("steps%d" % steps)
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--small", "--steps", str(steps), "--warmup", "1",
                            "--no-cpu-baseline", "--no-beam", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert p.returncode == 0, p.stderr[-2000:]
        line = lines[steps] = json.loads(p.stdout.strip().splitlines()[-1])
        assert sorted(os.listdir(out)) == ["tokens.npy"]          # --small has no denoise loop
        toks = dumped[steps] = np.load(out / "tokens.npy")
        assert toks.dtype == np.float64 and toks.shape == (1, 128)
        # the ids of the last timed step, as the JSON line hashes them
        assert hashlib.sha1(toks.astype(np.int64).tobytes()).hexdigest()[:16] == line["tokens_sha1"]
    # every timed generate launches the same kernels: the timed region holds exactly --steps of them
    assert lines[1]["gpu_launches"] > 0 and lines[3]["gpu_launches"] == 3 * lines[1]["gpu_launches"]
    assert np.array_equal(dumped[1], dumped[3])


@pytest.mark.gpu
def test_denoise_times_the_loops_it_is_asked_for(cuda):
    """run_denoise (the denoise half of c2, and c5) times `timed_loops` loops after `warm_loops` untimed ones: launches per
    Euler step, counted over the timed region and divided by timed_loops x steps, do not depend on timed_loops"""
    import bench
    eng, _ = bench.make_unet_engine()
    try:
        r1 = bench.run_denoise(steps=2, hw=32, warm_loops=1, timed_loops=1, eng=eng)
        r3 = bench.run_denoise(steps=2, hw=32, warm_loops=2, timed_loops=3, eng=eng)
    finally:
        eng.close()
    assert r1["launches_per_step"] > 0 and r3["launches_per_step"] == r1["launches_per_step"]
    assert r1["finite"] and r3["latents_sha1"] == r1["latents_sha1"]
