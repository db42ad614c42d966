"""bench.py --dump-outputs: the results of the last timed train and eval steps as float .npy files, the same from run
to run with the same arguments (a small catalog and a few steps keep the two runs short)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = ["--items", "3000", "--steps", "3", "--warmup", "1", "--no_kernels", "--no_cpu_baseline", "--loop_sessions", "0"]


def run_bench(out):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *ARGS, "--dump-outputs", str(out)],
                         capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    return line, {f[:-4]: np.load(os.path.join(out, f)) for f in sorted(os.listdir(out))}


def test_dump_outputs_hold_the_last_timed_steps_and_repeat(tmp_path):
    line, got = run_bench(tmp_path / "a")
    assert line["steps"] == 3 and len(line["ms_per_step_spread"]["first_ms"]) == 3
    assert all(v.dtype in (np.float32, np.float64) for v in got.values())
    assert sum(v.nbytes for v in got.values()) <= 64 << 20
    assert got["train_loss"].shape == (512,) and np.isfinite(got["train_loss"]).all()
    np.testing.assert_allclose(got["train_loss"].mean(), line["loss_last_step"], rtol=1e-5)
    assert got["item_rows"].shape == (len(got["item_row_ids"]), 250) and "param_W_p" in got
    ids = got["eval_top20_ids"]
    assert ids.shape == (512, 20) and (ids >= 0).all() and (ids < 3000).all() and (ids == np.round(ids)).all()
    assert got["eval_n_greater"].shape == got["eval_cross_loss"].shape == (512,)
    _, again = run_bench(tmp_path / "b")
    assert again.keys() == got.keys()
    for k, v in got.items():
        np.testing.assert_allclose(again[k], v, rtol=1e-5, atol=1e-7, err_msg=k)
