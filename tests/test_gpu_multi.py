"""Real multi-GPU parity of the partitioned pipelines (needs >= 2 visible B200s; skipped on a 1-GPU box).

Launches tools/check_partitions.py under torchrun at every even world size the box offers (2, 4, 8): 1-D phased and
2-D on the same seeded graph, every result compared with the plain all-gather + one-launch aggregation, which runs
last (see the tool's header).
"""
import json
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.timeout(900)
@pytest.mark.parametrize("world", [2, 4, 8])
def test_partitions_agree_on_real_gpus(world):
    n_gpus = torch.cuda.device_count()
    if n_gpus < world:
        pytest.skip(f"needs {world} GPUs, {n_gpus} visible")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tools", "check_partitions.py"), "--nodes", "1000003", "2000000"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=850, cwd=ROOT)
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith('{"check"')]
    assert out.returncode == 0 and lines, out.stdout[-2000:] + out.stderr[-2000:]
    rep = json.loads(lines[-1])
    assert rep["ok"] and len(rep["graphs"]) == 2
    for graph in rep["graphs"]:
        assert set(graph["results"]) >= {"1d-plain", "1d-phased", "2d"}
        for name, res in graph["results"].items():
            assert res["y_max_err_rel"] <= 5e-6 and res["counters_equal"], (name, res)
