"""N > 1: world_size-2 (and 4) `gloo` runs on CPU for the host logic, and the
real NCCL path when the box has >= 2 GPUs."""
import os
import socket
import subprocess
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))


def _free_port():
    # a port picked by the kernel, not a fixed number: other jobs on the host may hold any
    # given one.  Not race-free: the socket is closed before torchrun binds the port, and
    # another process may take it in between.
    with socket.socket(socket.AF_INET, socket.SOCK_STREAM) as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _run(mode, nproc, tmp_path):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(HERE, "mp_worker.py"), mode]
    env = dict(os.environ, OMP_NUM_THREADS="1", PA_TEST_SCRATCH=str(tmp_path))
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    errs = [l for l in out.stderr.splitlines() if l.startswith("WORKER-ERROR")]
    assert out.returncode == 0, "\n".join(errs[-60:]) + out.stdout[-1500:] + out.stderr[-1500:]
    assert f"MP_WORKER_OK mode={mode} world={nproc}" in out.stdout, out.stdout[-2000:]
    return out.stdout


@pytest.mark.parametrize("nproc", [2, 4])
def test_gloo_host_logic(nproc, tmp_path):
    _run("gloo", nproc, tmp_path)


@pytest.mark.gpu
@pytest.mark.parametrize("nproc", [2, 4, 5, 6, 8])
def test_ipc_transpose_ranks_sharing_gpus(nproc, tmp_path):
    """The whole multi-rank path on ANY box, a single-GPU one included: `nproc`
    processes (round-robin over the visible GPUs) joined by the NCCL-free
    communicator -- CUDA-IPC windows, NVLink/peer flag words, the one-launch
    multi-peer put/get kernels and the library's own staged exchange."""
    _run("ipc", nproc, tmp_path)


@pytest.mark.gpu
@pytest.mark.parametrize("nproc", [2, 4, 8])
def test_nccl_transpose(nproc, tmp_path):
    if torch.cuda.device_count() < nproc:
        pytest.skip(f"needs {nproc} GPUs")
    _run("nccl", nproc, tmp_path)
