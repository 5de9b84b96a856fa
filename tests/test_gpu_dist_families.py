"""GPU: data-parallel IPR-SRGAN and IPR-CycleGAN steps (two ranks, ``torch.distributed.run``) against single-process
references (tests/family_dist_worker.py):

* SRGAN, the same shard on both ranks: metrics and parameters bit-identical to one trainer on that shard -- the
  reduced gradient (g + g) / 2 and the reduced metrics are exact;
* SRGAN, different shards: metrics within 1e-4 of two replicas in one process whose gradients are averaged before
  each Adam step, replicas bit-identical to each other;
* CycleGAN, 2 ranks x batch 1: the trainer at batch 2 on the whole batch (InstanceNorm has no cross-sample
  statistics), image pools queried with the gathered batch: same pool counts, the rest within the bf16 budget.

Every rank returns the same metrics dict.  With NCCL (one GPU per rank, eager and CUDA graph) the tests need two
GPUs; the gloo variant puts both ranks on one GPU (eager: gloo collectives cannot be captured)."""
import os
import signal
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKER = os.path.join(ROOT, "tests", "family_dist_worker.py")
KINDS = ["srgan_same", "srgan_diff", "cyclegan"]


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _run(cmd, timeout=900):
    """Run in a session of its own, so that a timeout takes every worker process down with the launcher."""
    p = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, start_new_session=True)
    try:
        out, err = p.communicate(timeout=timeout)
    except subprocess.TimeoutExpired:
        os.killpg(p.pid, signal.SIGKILL)
        out, err = p.communicate()
        pytest.fail("timed out: %s\n%s\n%s" % (" ".join(cmd), out[-3000:], err[-3000:]))
    assert p.returncode == 0, out[-3000:] + err[-3000:]


def _rel(a, b):
    return float((a - b).norm() / (b.norm() + 1e-12))


def _check(kind, mode, backend, tmp_path):
    ref_path, dist_path = str(tmp_path / "ref.pt"), str(tmp_path / "dist.pt")
    _run([sys.executable, WORKER, kind, mode, backend, ref_path])
    _run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
          "127.0.0.1", "--master-port", str(_free_port()), WORKER, kind, mode, backend, dist_path])
    ref, got = torch.load(ref_path), torch.load(dist_path)
    assert got["world"] == 2 and got["replicas_identical"]
    for m in got["rank_metrics"][1:]:
        assert m == got["rank_metrics"][0]                      # the same dict on every rank
    assert len(got["metrics"]) == len(ref["metrics"]) == 2
    if kind == "srgan_same":
        assert got["metrics"] == ref["metrics"]
        assert torch.equal(got["params"], ref["params"])
        assert got["launches"] == ref["launches"] and got["launches"] > 0    # the collectives add no library launch
        return
    tol = 1e-4 if kind == "srgan_diff" else 2e-2
    for g, w in zip(got["metrics"], ref["metrics"]):
        assert sorted(g) == sorted(w)
        for k in w:
            assert abs(g[k] - w[k]) <= tol * max(1.0, abs(w[k])), (k, g[k], w[k])
    if kind == "cyclegan":
        assert got["pools_identical"]
        for (cg, ig), (cr, ir) in zip(got["pool"], ref["pool"]):
            assert float(cg) == float(cr) == 4.0                  # full after step 2, exchanging in step 3
            # the stored images come from steps 1-3: after the first Adam step, which moves every weight by about
            # +-lr whatever the size of its gradient, bf16-level gradient differences are weight differences of up to
            # 2 lr, and the images generated next inherit them (measured 0.034 on a B200; one forward alone: 3e-2,
            # tests/test_gpu_srgan_cyclegan.py)
            assert ig.shape == ir.shape and _rel(ig, ir) <= 5e-2
        assert float((got["params"] - ref["params"]).abs().max()) <= 2e-3


@pytest.mark.parametrize("mode", ["eager", "graph"])
@pytest.mark.parametrize("kind", KINDS)
def test_two_rank_family_step_nccl(kind, mode, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _check(kind, mode, "nccl", tmp_path)


@pytest.mark.parametrize("kind", KINDS)
def test_two_rank_family_step_gloo_one_gpu(kind, tmp_path):
    _check(kind, "eager", "gloo", tmp_path)
