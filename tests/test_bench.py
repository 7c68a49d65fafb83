"""bench.py's command line: argument refusals (CPU) and --dump-outputs (GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*argv):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], capture_output=True, text=True,
                          timeout=900)


@pytest.mark.parametrize("argv,flag", [(["--steps", "0"], "--steps"),
                                       (["--impl", "reference", "--dump-outputs", "d"], "--dump-outputs")])
def test_refusals_name_the_flag(argv, flag):
    r = _bench(*argv)
    assert r.returncode == 2 and flag in r.stderr, r.stderr


@pytest.mark.gpu
def test_dump_outputs_of_two_runs_agree(tmp_path):
    """The fixture workload (K = 5,830: W1 fits the sample whole, 13 steps per epoch).  Two runs of 3 + 5 steps, which
    end inside the first epoch, dump the same arrays; a run of 3 + 20 steps, across an epoch end, dumps arrays of the
    same names and shapes.  Every array is float32 and non-empty, the whole dump at most 64 MB."""
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    dumps = []
    for run, (steps, warmup) in enumerate([(5, 3), (5, 3), (20, 3)]):
        d = tmp_path / f"run{run}"
        r = _bench("--gpus", "1", "--steps", str(steps), "--warmup", str(warmup), "--workload", "fixture",
                   "--dump-outputs", str(d), "--no-queue", "--no-large-batch", "--no-cpu-baseline", "--group", "0",
                   "--e2e-epochs", "1")
        assert r.returncode == 0, r.stderr[-4000:]
        line = json.loads([s for s in r.stdout.splitlines() if s.startswith("{")][-1])
        assert line["steps"] == steps and line["warmup"] == warmup
        dumps.append({f[:-4]: np.load(d / f) for f in sorted(os.listdir(d))})
    a, b, c = dumps
    assert {k: v.shape for k, v in a.items()} == {k: v.shape for k, v in b.items()} == {k: v.shape for k, v in c.items()}
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert all(v.dtype == np.float32 and v.size > 0 for v in a.values())
    assert a["w04_dense01_kernel_sampled_rows"].shape == (5830, 256)
    assert a["w00_bn_gamma"].shape == (5830,) and a["w27_dense12_bias"].shape == (2,)
    assert np.isfinite(a["last_loss"]).all()
    for name in a:
        np.testing.assert_array_equal(a[name], b[name], err_msg=name)
