"""GPU: `bench.py --dump-outputs` writes the same outputs on every run with the same arguments, so that two builds can
be compared output for output.  The timed step scatters with float atomics; the dumped last step restarts from the
seeded state, so two runs may differ by rounding only."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import assert_close

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _dump(out):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--batch", "65536", "--steps", "6",
           "--warmup", "3", "--quick", "--no-topn", "--no-models", "--no-bands", "--dump-outputs", str(out)]
    subprocess.run(cmd, check=True, stdout=subprocess.DEVNULL, env=dict(os.environ, PYTHONDONTWRITEBYTECODE="1"))
    return {n[:-4]: np.load(os.path.join(str(out), n)) for n in sorted(os.listdir(str(out)))}


def test_bench_dump_is_the_same_on_every_run(cuda, tmp_path):
    a, b = _dump(tmp_path / "a"), _dump(tmp_path / "b")
    assert sorted(a) == ["feature_bias", "feature_embeddings", "loss"]
    assert all(v.dtype == np.float32 for v in a.values())
    assert a["feature_embeddings"].shape == (5382, 64)
    assert a["loss"][0] == b["loss"][0]             # the forward pass from the seeded weights has no atomics
    assert_close(b["feature_embeddings"], a["feature_embeddings"], what="dumped weights of two runs")
    assert np.array_equal(a["feature_bias"], b["feature_bias"])
