"""bench.py --dump-outputs: the arrays written are the landmarks and scores the timed path computed in its last step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def _bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), capture_output=True, text=True,
                          timeout=900, cwd=ROOT)


@pytest.mark.parametrize("args", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_rejects_bad_arguments(args):
    out = _bench(*args)
    assert out.returncode == 2, out.stderr[-2000:]


@pytest.mark.gpu
def test_bench_dumps_last_timed_step(tmp_path):
    import frames
    from peppa_pig_face_landmark_b200 import ONNXEngine
    B, steps = 8, 2
    runs = []
    for k in range(2):
        d = tmp_path / ("run%d" % k)
        out = _bench("--steps", str(steps), "--warmup", "1", "--batch", str(B), "--no-pipeline", "--no-cpu-baseline",
                     "--dump-outputs", str(d))
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == steps
        runs.append({n: np.load(d / (n + ".npy")) for n in ("landmarks", "scores")})
    lm, sc = runs[0]["landmarks"], runs[0]["scores"]
    assert lm.dtype == sc.dtype == np.float32 and lm.shape == (B, 196) and sc.shape == (B, 98)
    for n in runs[0]:
        assert np.array_equal(runs[0][n], runs[1][n]), n            # same arguments, same inputs, same outputs
    # the last of `steps` timed steps runs input set (steps - 1) of the 4 rotated seeded sets (bench.py: seed 100 + set)
    crops = frames.noise_crops(B, seed=100 + (steps - 1))
    eng = ONNXEngine(os.path.join(ROOT, "peppa_pig_face_landmark_b200", "pretrained", "kps_student.onnx"), max_batch=B)
    rlm, rsc = eng.run_u8(crops)
    assert np.array_equal(lm, rlm) and np.array_equal(sc, rsc)
