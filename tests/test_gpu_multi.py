"""GPU: the data-parallel exchange end to end (tools/check_multigpu.py under torch.distributed.run):
fused exchange launch vs sh_backward + one NCCL all-reduce of the flat buffer, replicas bit-identical after Adam
steps, and both again after a lock-step change of the Gaussian count (odd N).
 * world size 1 runs everywhere (symmetric memory, re-binding of the gradient buffer, both CTA roles of the launch,
   resize) -- the driver's 1-GPU box included;
 * world size 2 needs two devices (skipped otherwise), once with the NVSwitch multimem
   all-reduce role and once with the peer-pointer one."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(nproc, port, env=None):
    e = dict(os.environ)
    e.update(env or {})
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc),
                        "--master-addr", "127.0.0.1", "--master-port", str(port),
                        os.path.join(ROOT, "tools", "check_multigpu.py")], capture_output=True, text=True, timeout=600,
                       env=e)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-2000:])
    assert "fused_ok=True" in r.stdout and "replicas_in_sync=True" in r.stdout and "after_resize_ok=True" in r.stdout
    return r.stdout


def test_fused_exchange_world1_end_to_end():
    _run(1, 29531)


def test_fused_exchange_matches_nccl_allreduce_2gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    out = _run(2, 29533)
    out2 = _run(2, 29535, {"GSB_EXCHANGE_MULTICAST": "0"})
    assert "multicast=False" in out2
