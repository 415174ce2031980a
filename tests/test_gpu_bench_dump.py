"""bench.py --dump-outputs: the last timed step's outputs as float32 / float64 .npy files, the same from run to run."""
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_dump(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "2",
                        "--vocab", "100000", "--batch", "1024", "--no-extras", "--no-cpu-baseline",
                        "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=280)
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout)["steps"] == steps
    return {os.path.basename(p)[:-4]: np.load(p) for p in glob.glob(os.path.join(out_dir, "*.npy"))}


@pytest.mark.gpu
def test_dump_outputs_repeat_exactly_and_follow_steps(tmp_path):
    a, b = _bench_dump(tmp_path / "a", 5), _bench_dump(tmp_path / "b", 5)
    assert {"loss_terms", "prob", "sample_rows", "fm_v_sample_rows", "fm_w_sample_rows", "fm_bias"} <= a.keys() == b.keys()
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for name in a:
        assert a[name].dtype in (np.float32, np.float64), name
        np.testing.assert_array_equal(a[name], b[name], err_msg=name)
    assert a["loss_terms"].shape == (3,) and (a["loss_terms"] > 0).all()
    assert a["fm_v_sample_rows"].shape == (a["sample_rows"].size, 16) and a["prob"].shape == (1024,)
    # one more timed step is one more optimizer step on the same inputs: the state must differ
    c = _bench_dump(tmp_path / "c", 6)
    assert not np.array_equal(a["fm_bias"], c["fm_bias"])
