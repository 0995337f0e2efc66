"""Expert-parallel prefill vs the single-GPU model with identical weights; needs >= 2 GPUs (skips on one).
  seq : sequence-sharded dense part + all-gathered K/V and routed rows + fused P2P combine (default; bit-identical)
  p2p : replicated dense part, the down-projection GEMM epilogue pushes rows to the token owners (bit-identical)
  nccl: partial sums + one NCCL all-reduce per layer (library baseline, statistical bound)"""
import os
import subprocess
import sys
from pathlib import Path

import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent


@pytest.mark.gpu
@pytest.mark.parametrize("mode,port", [("seq", 29532), ("p2p", 29533), ("nccl", 29534)])
def test_ep2_prefill_matches_single_gpu(mode, port):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(port), str(ROOT / "tests" / "ep_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, VITA_B200_EP=mode))
    print(res.stdout[-2000:], res.stderr[-2000:])
    assert res.returncode == 0
