"""bench.py --dump-outputs: the decision table of one cycle as float64 .npy files, exact for every value the C ABI returns."""
import os
import subprocess
import sys

import numpy as np

import bench
from kube_batch_b200 import abi, engine


def test_dump_outputs_writes_every_decision_field_exactly(tmp_path):
    dec = np.zeros(4, dtype=np.dtype(abi.DECISION_DTYPE))
    dec["node"] = [-1, 0, 7, 2**31 - 1]
    dec["kind"] = [abi.KB_KIND_NONE, abi.KB_KIND_ALLOCATED, abi.KB_KIND_PIPELINED, abi.KB_KIND_SKIPPED]
    dec["dispatched"] = [0, 1, 1, 0]
    dec["step"] = [0xFFFFFFFF, 0, 1, 2]
    dec["dispatch_step"] = [0xFFFFFFFF, 3, 3, 0]
    out = tmp_path / "out"
    bench.dump_outputs(str(out), engine.CycleResult(dec, abi.kb_stats()))
    assert sorted(os.listdir(out)) == sorted(f"decisions_{f}.npy" for f in bench.DECISION_FIELDS)
    for f in bench.DECISION_FIELDS:
        a = np.load(out / f"decisions_{f}.npy")
        assert a.dtype == np.float64
        np.testing.assert_array_equal(a, dec[f].astype(np.int64), err_msg=f)


def test_steps_below_one_are_refused():
    p = subprocess.run([sys.executable, bench.__file__, "--steps", "0"], capture_output=True, text=True)
    assert p.returncode == 2 and "--steps" in p.stderr
