"""Synchronised BatchNorm across data-parallel ranks on real GPUs (needs >= 2 visible devices, skips otherwise):
launches tests/dp_sync_bn_worker.py with torch.distributed.run, one process per GPU over NCCL.  Per-rank batches of 512
rows take the bf16 route whose GEMM accumulates the statistics (k_bn_act_pre), 8192 rows the k_bn_finalize route; the
fp32-parity path always takes k_bn_finalize.  The unequal case (512 + 300 rows) checks that the counts travel with the
moments.  With one GPU both ranks share it (CUDA IPC within the device, gloo rendezvous)."""
import json
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("path,n0,n1", [("bf16", 512, 512), ("bf16", 8192, 8192), ("fp32", 512, 512),
                                        ("fp32", 8192, 8192), ("fp32", 512, 300)])
def test_sync_batch_norm_matches_one_gpu_on_the_global_batch(path, n0, n1):
    if torch.cuda.device_count() < 1:
        pytest.skip("needs a GPU")
    world = 2
    env = dict(os.environ)
    if torch.cuda.device_count() < 2:        # both ranks on one device: the protocol and the arithmetic, not NVLink
        env["LCN_DP_SHARE_GPU"] = "1"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", "29547", os.path.join(ROOT, "tests", "dp_sync_bn_worker.py"),
           path, str(n0), str(n1)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=420, cwd=ROOT, env=env)
    lines = [json.loads(l) for l in r.stdout.splitlines() if l.startswith("{")]
    if os.environ.get("LCN_RECORD_DIR"):      # keep the per-rank records (errors, trajectories) of the run
        with open(os.path.join(os.environ["LCN_RECORD_DIR"], f"dp_sync_bn_{path}_{n0}_{n1}.json"), "w") as f:
            json.dump(lines, f, indent=1)
    assert r.returncode == 0, json.dumps(lines, indent=1)[-4000:] + r.stderr[-3000:]
    assert len(lines) == world and all(l["taps_identical"] and not l["fails"] for l in lines)
