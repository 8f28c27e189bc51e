"""Multi-GPU parity of the row-partitioned GAT and GATv2 models (LargeGraphAttentionModel): the
exchange of the layer GEMM's output (both transports) under torchrun on up to four GPUs of the box,
checked against the float64 restatements by tests/run_large_attn_multi_gpu.py --conv.  Skips on a
box with fewer than two GPUs."""
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
@pytest.mark.parametrize("conv", ["gat", "gatv2"])
def test_attention_halo_exchange_matches_float64(conv, transport):
    import torch

    n_gpus = torch.cuda.device_count()
    if n_gpus < 2:
        pytest.skip("needs at least two GPUs")
    world = min(n_gpus, 4)
    port = 29500 + (os.getpid() + 13 * world + 5 * len(conv) + len(transport) + 700) % 2000
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           str(ROOT / "tests" / "run_large_attn_multi_gpu.py"), "--nodes", str(NODES),
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
    heads = 4
    assert res["stats"]["exchanged_floats_per_halo_row"] == [128 + 2 * heads if conv == "gat" else 128] * 2
    n = NODES - NODES % world
    assert 0 < res["stats"]["halo_rows"] <= n * (world - 1) // world
