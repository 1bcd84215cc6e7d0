"""GPU parity of the row-sharded multi-GPU path (needs >= 2 GPUs: `gpurun --gpus 2`): W ranks with
row-sharded tables and NCCL all-to-alls must reproduce the single-GPU trainer on the global batch."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
HERE = os.path.dirname(os.path.abspath(__file__))


def _run(n, *args, port=29731):
    if not torch.cuda.is_available() or torch.cuda.device_count() < n:
        pytest.skip(f"needs >= {n} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(HERE, "sharded_worker.py"), *args]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=400)
    print(r.stdout[-6000:])
    print(r.stderr[-3000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "FAIL" not in r.stdout


@pytest.mark.parametrize("mode", ["eager", "graph"])
def test_sharded_matches_single_gpu(mode):
    """fp32 parity mode, W = 2: losses, dense parameters and table shards after 3 steps equal the single-GPU
    trainer on the global batch (1e-5); checkpoints W -> W, W -> 1, 1 -> W bit-exact."""
    _run(2, mode, "f32", "96", "auto")


@pytest.mark.parametrize("n", [2, 8])
@pytest.mark.parametrize("cap", ["auto", "tight"])
def test_sharded_benchmarked_path(n, cap):
    """THE benchmarked multi-GPU combination: bf16 activations + tcgen05 kernels + peer-memory gather / scatter +
    the whole step in one CUDA graph, at W = 2 and W = 8, with the default bucket capacity and with buckets filled
    to the last slot; against the same-dtype single-GPU trainer on the global batch; first-step gather bit-exact."""
    _run(n, "graph", "bf16", "512", cap, port=29741 + n)


@pytest.mark.parametrize("n", [2, 8])
def test_sharded_forced_overflow_is_reported(n):
    """One slot too few for the fullest bucket: the step must not hang or corrupt silently — check_overflow() raises."""
    _run(n, "graph", "bf16", "512", "overflow", port=29761 + n)


@pytest.mark.parametrize("n", [2, 8])
@pytest.mark.parametrize("which,mode", [("autoint", "eager"), ("autoint", "graph"), ("video_dnn", "eager"), ("video_dnn", "graph")])
def test_sharded_composed_models(n, which, mode):
    """BASELINE configs[3] / configs[4] on W GPUs: AUTOINT (rank/multi_head) and mtl_net (staytime VideoDnn) over the
    row-sharded ShardedEmbeddingFeatures (Adam and AdaGrad, single-valued and sequence columns) with data-parallel
    dense parts, against the single-GPU model on the global batch: first lookup bit-exact, losses / global table /
    dense parameters after 3 steps at 1e-5; eagerly and as one CUDA graph per step."""
    if not torch.cuda.is_available() or torch.cuda.device_count() < n:
        pytest.skip(f"needs >= {n} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", str(29781 + n), os.path.join(HERE, "sharded_models_worker.py"),
           which, mode]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=400)
    print(r.stdout[-4000:])
    print(r.stderr[-3000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "FAIL" not in r.stdout
