"""
PeerResultRing (setk_b200/distributed.py): results reach rank 0 by device-to-peer copies through a
mapping of rank 0's buffer (torch symmetric memory; legacy CUDA IPC as the fallback), no collective
kernel.  Two processes exercise the mappings, the side-stream ordering and the slot arithmetic; `bench.py --gpus N` checks the same thing across
GPUs (checksums of every rank's last batch).
"""
import os
import socket
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.gpu
def test_peer_ring_two_processes_one_gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, os.path.join(HERE, "peer_ring_worker.py")], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = []
    for p in procs:
        try:
            out, _ = p.communicate(timeout=300)
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            raise
        outs.append(out)
    assert all(p.returncode == 0 for p in procs), "\n----\n".join(o[-3000:] for o in outs)
