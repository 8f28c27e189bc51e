"""Multi-GPU parity of the row-partitioned GIN, SAGE and PNA models: the halo exchange (both
transports) under torchrun on up to four GPUs of the box, checked against the CPU oracle by
tests/run_large_model_multi_gpu.py --conv.  Skips on a box with fewer than two GPUs."""
import json
import os
import subprocess
import sys
from pathlib import Path

import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
NODES = 40000


@pytest.mark.parametrize("transport", ["nccl", "p2p"])
@pytest.mark.parametrize("conv", ["gin", "sage", "pna"])
def test_halo_exchange_matches_the_oracle(conv, transport):
    import torch

    n_gpus = torch.cuda.device_count()
    if n_gpus < 2:
        pytest.skip("needs at least two GPUs")
    world = min(n_gpus, 4)
    port = 29500 + (os.getpid() + 11 * world + 3 * len(conv) + len(transport)) % 2000
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           str(ROOT / "tests" / "run_large_model_multi_gpu.py"), "--nodes", str(NODES),
           "--transport", transport, "--conv", conv]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=str(ROOT))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert lines, r.stdout[-2000:]
    res = json.loads(lines[-1])
    assert res["ok"], res
    assert res["conv"] == conv and res["stats"]["transport"] == transport
    assert res["err_out"] < 1e-4 and res["err_emb"] < 1e-4
    assert res["bit_identical_rerun"]
    # a true halo: fewer rows than the full remote set travel
    n = NODES - NODES % world
    assert 0 < res["stats"]["halo_rows"] <= n * (world - 1) // world
