"""The collective evaluate() of the row-sharded trainer (needs >= 2 GPUs): per-rank streams of unequal length, zero
batches on some ranks, against the single-GPU evaluate() of the concatenated stream from the same checkpoint."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.parametrize("n", [2, 8])
@pytest.mark.parametrize("mode,dtype", [("graph", "bf16"), ("eager", "f32")])
def test_sharded_evaluate_matches_single_gpu(n, mode, dtype):
    if not torch.cuda.is_available() or torch.cuda.device_count() < n:
        pytest.skip(f"needs >= {n} GPUs")
    port = 29801 + n + (10 if dtype == "f32" else 0)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(HERE, "sharded_eval_worker.py"),
           mode, dtype, "256"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=400)
    print(r.stdout[-6000:])
    print(r.stderr[-3000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "FAIL" not in r.stdout and "PASS" in r.stdout
