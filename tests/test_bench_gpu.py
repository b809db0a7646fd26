"""GPU: bench.py --dump-outputs writes what the last timed step computed (a one-block text run of the 8B shape)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_dump(tmp_path, out):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
           "--workload", "text", "--layers", "1", "--batch", "1", "--seq", "256", "--no-cpu-baseline",
           "--no-int8-peak", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=tmp_path, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_dump_outputs_of_the_last_timed_step(tmp_path):
    out = tmp_path / "dump"
    line = _bench_dump(tmp_path, out)
    assert line["steps"] == 2
    assert sorted(os.listdir(out)) == ["text_grads.npy", "text_loss.npy"]
    loss, grads = np.load(out / "text_loss.npy"), np.load(out / "text_grads.npy")
    assert loss.dtype == np.float32 and loss.shape == () and round(float(loss), 4) == line["loss"]
    # every trainable gradient of one block: LoRA r=8 on the seven projections, the two block norms, the final norm
    D, KV, F = 4096, 1024, 14336
    lora = 8 * ((D + D) * 2 + (D + KV) * 2 + (D + F) * 3)
    assert grads.dtype == np.float32 and grads.shape == (lora + 3 * D,)
    assert np.isfinite(grads).all() and np.count_nonzero(grads) > grads.size // 2
    # a second run with the same arguments computes the same outputs: the inputs of every step are the seeded ones, and
    # the only run-to-run freedom is the order of float atomics inside one step (bf16 gradients: a few ulp at most)
    _bench_dump(tmp_path, tmp_path / "again")
    loss2, grads2 = np.load(tmp_path / "again" / "text_loss.npy"), np.load(tmp_path / "again" / "text_grads.npy")
    assert abs(float(loss2) - float(loss)) <= 1e-5 * abs(float(loss))
    assert np.abs(grads2 - grads).max() <= 1e-2 * np.abs(grads).max()
