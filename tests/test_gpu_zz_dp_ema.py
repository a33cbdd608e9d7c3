"""Data-parallel training of the EMA-codebook variant on 2 GPUs: scripts/check_dp_ema.py under torch.distributed.run (the
EMA step over the global batch bit-identical to the single-device step, replicas, resets, the trainer against the
unmodified reference), and the index_improve CLI under torchrun."""
import glob
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
two_gpus = pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _torchrun(*argv, nproc=2, timeout=1800, cwd=ROOT):
    return subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc), "--master-addr",
                           "127.0.0.1", "--master-port", str(_free_port()), *argv],
                          capture_output=True, text=True, timeout=timeout, cwd=cwd)


@pytest.mark.parametrize("nproc", [pytest.param(1), pytest.param(2, marks=two_gpus)])
def test_dp_ema_equals_single_device_step(nproc):
    """nproc 1 runs the same path (publish into the one symmetric buffer, gather from it, EMA kernel) on a single GPU."""
    r = _torchrun(os.path.join(ROOT, "scripts", "check_dp_ema.py"), "--no-timing", nproc=nproc)
    assert r.returncode == 0, r.stderr[-3000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["failures"] == [] and out["ok"], out
    assert all(out["op_cases"].values()) and out["reset"]
    t = out["trainer"]
    assert t["reference"]["ok"] and t["replicas_equal"] and t["first_step_ema_buffers_bitwise"]
    assert t["reset_interval_3"]["ok"] and t["reset_interval_3"]["codes_reset_single_device"] > 0 and out["world"] == nproc
    assert t["empty_rank"]["ok"] and t["kmeans_init"]["ok"] and t["batchnorm"]["ok"]


@two_gpus
def test_index_improve_cli_trains_on_two_gpus(tmp_path):
    """torchrun -m lcrec_b200.index_improve.main: 2 epochs on a small seeded .npy; rank 0's checkpoint loads into a
    single-device RQVAE of the variant with finite EMA buffers."""
    from lcrec_b200.index_improve.models import RQVAE
    x = np.random.default_rng(5).standard_normal((400, 128)).astype(np.float32)
    path = str(tmp_path / "emb.npy")
    np.save(path, x)
    ckpt = tmp_path / "ckpt"
    r = _torchrun("-m", "lcrec_b200.index_improve.main", "--data_path", path, "--num_emb_list", "32", "32", "32",
                  "--e_dim", "16", "--layers", "64", "48", "--batch_size", "100", "--epochs", "2", "--eval_step", "2",
                  "--num_workers", "0", "--kmeans_iters", "10", "--reset_interval", "3", "--warmup_epochs", "1",
                  "--ckpt_dir", str(ckpt), timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    found = glob.glob(str(ckpt / "*" / "best_loss_model.pth"))
    assert len(found) == 1, found
    state = torch.load(found[0], map_location="cuda:0", weights_only=False)["state_dict"]
    m = RQVAE(in_dim=128, num_emb_list=[32] * 3, e_dim=16, layers=[64, 48], kmeans_init=True, sk_epsilons=[0.0] * 3)
    m.load_state_dict(state)
    for q in m.rq.vq_layers:
        assert torch.isfinite(q._ema_cluster_size).all() and torch.isfinite(q._ema_w).all()
        assert float(q._ema_cluster_size.sum()) > 0
