"""Multi-GPU parity (needs >= 2 GPUs on the box; skipped otherwise)."""
import os
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("peer", ["", "1"])
def test_point_sharded_solve_matches_single_gpu(peer):
    """peer = "1": the all-reduces go through NVLink peer memory (csrc/peer_reduce.cuh, LCBA_PEER_REDUCE=1)
    instead of ncclAllReduce; the worker checks the same parity and that the route really is the peer one."""
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ws = 2 if n < 4 else 4
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(ws),
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(REPO, "tests", "_gpu_dist_worker.py")]
    env = dict(os.environ, LCBA_PEER_REDUCE=peer, LCBA_PEER_VERBOSE="1")
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    for r in range(ws):
        assert "rank %d ok" % r in out.stdout
        route = "rank %d/%d: peer all-reduce on" % (r, ws)
        assert (route in out.stderr) == (peer == "1"), out.stderr[-2000:]
