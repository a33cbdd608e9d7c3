"""End-to-end time of the generate_indices CLI on 1, 2 and 8 GPUs of one box (fp16 and fp32 .npy in the page cache).

    python scripts/probe_generate_dist.py --items-per-gpu 1000000 --gpus 1 2 8 --out probe.jsonl

For every (dtype, GPU count): a seeded checkpoint of the run.sh architecture (4096 -> ... -> 32, 4 x 256 codes), a .npy of
items-per-gpu x GPUs synthetic items (written once, then read once so that it sits in the page cache), and one CLI run -
plain on 1 GPU, under torchrun on more - with LCREC_DIST_TIMING=1, which makes the CLI print its phases: PASS-0 streaming,
exchange and rounds (CUDA events of generate_codes_sharded; on one GPU the rounds are the library's stage events of the
collision checks and Sinkhorn, and PASS-0 streaming the rest of generate_codes), JSON formatting and the file write.  One JSON
line per run, with the card name and its power limit (both are part of the number).  Writes only under --workdir and --out.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
DIMS = [4096, 2048, 1024, 512, 256, 128, 64, 32]


def _card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                               text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def _checkpoint(path):
    import argparse as ap
    import torch
    from lcrec_b200.models.rqvae import RQVAE
    from lcrec_b200.synth import seeded_weights
    ws, bs, cbs = seeded_weights(DIMS, [256] * 4, 32, seed=3, cb_scale=0.02)
    m = RQVAE(in_dim=DIMS[0], num_emb_list=[256] * 4, e_dim=32, layers=DIMS[1:-1], sk_epsilons=[0.0, 0.0, 0.0, 0.003], sk_iters=50)
    sd = m.state_dict()
    lin = sorted([k for k in sd if k.startswith("encoder.mlp_layers.") and k.endswith(".weight")], key=lambda s: int(s.split(".")[2]))
    for k, w, b in zip(lin, ws, bs):
        sd[k] = torch.from_numpy(w); sd[k.replace(".weight", ".bias")] = torch.from_numpy(b)
    for l, cb in enumerate(cbs):
        sd[f"rq.vq_layers.{l}.embedding.weight"] = torch.from_numpy(cb)
    args = ap.Namespace(data_path="unused.npy", num_emb_list=[256] * 4, e_dim=32, layers=DIMS[1:-1], dropout_prob=0.0, bn=False,
                        loss_type="mse", quant_loss_weight=1.0, kmeans_init=False, kmeans_iters=100, sk_epsilons=[0.0, 0.0, 0.0, 0.003],
                        sk_iters=50)
    torch.save({"args": args, "state_dict": sd}, path)


def _items(path, n, dtype):
    from lcrec_b200.synth import synth_items
    out = np.lib.format.open_memmap(path, mode="w+", dtype=dtype, shape=(n, DIMS[0]))
    step = 65536
    for s in range(0, n, step):
        out[s:s + step] = synth_items(min(step, n - s), DIMS[0], n_parents=max(n // 8, 1), seed=7, start=s)
    out.flush()
    del out
    with open(path, "rb") as f:                                  # into the page cache
        while f.read(1 << 26):
            pass


def _free_port():
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _run(ckpt, data, outdir, gpus, chunk_rows):
    cli = ["--ckpt_path", ckpt, "--data_path", data, "--output_dir", outdir, "--dataset", "Probe", "--chunk_rows", str(chunk_rows)]
    env = dict(os.environ, LCREC_DIST_TIMING="1")
    if gpus == 1:
        cmd = [sys.executable, "-m", "lcrec_b200.generate_indices", *cli]
    else:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(gpus), "--master-addr", "127.0.0.1",
               "--master-port", str(_free_port()), "-m", "lcrec_b200.generate_indices", *cli]
    t0 = time.perf_counter()
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT, env=env, timeout=3600)
    wall = time.perf_counter() - t0
    if r.returncode != 0:
        raise RuntimeError(r.stderr[-3000:])
    phases = {}
    for line in r.stderr.splitlines():
        if line.startswith("generate timing: "):
            phases = json.loads(line[len("generate timing: "):])
    return wall, phases


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--items-per-gpu", type=int, default=1_000_000)
    ap.add_argument("--gpus", type=int, nargs="+", default=[1, 2, 8])
    ap.add_argument("--dtypes", nargs="+", default=["float16", "float32"])
    ap.add_argument("--chunk_rows", type=int, default=131072)
    ap.add_argument("--workdir", default=None, help="where the .npy and the JSON go (default: a temporary directory)")
    ap.add_argument("--out", default=None, help="append the JSON lines here as well")
    a = ap.parse_args()
    import torch
    visible = torch.cuda.device_count()
    card, limit = _card()
    work = a.workdir or tempfile.mkdtemp(prefix="lcrec_probe_")
    try:
        ckpt = os.path.join(work, "ckpt.pth")
        _checkpoint(ckpt)
        for dtype in a.dtypes:
            for g in a.gpus:
                if g > visible:
                    continue
                n = a.items_per_gpu * g
                data = os.path.join(work, f"items_{dtype}_{n}.npy")
                _items(data, n, np.dtype(dtype))
                wall, phases = _run(ckpt, data, os.path.join(work, "out"), g, a.chunk_rows)
                inner = phases.get("codes_s", 0.0) + phases.get("json_s", 0.0) + phases.get("write_s", 0.0)
                line = {"gpus": g, "dtype": dtype, "items": n, "in_dim": DIMS[0], "chunk_rows": a.chunk_rows, "wall_s": round(wall, 3),
                        "items_per_s_wall": round(n / wall), "items_per_s_generate": round(n / inner) if inner else None,
                        "phases": phases, "card": card, "power_limit": limit}
                print(json.dumps(line), flush=True)
                if a.out:
                    with open(a.out, "a") as f:
                        f.write(json.dumps(line) + "\n")
                os.remove(data)
    finally:
        if a.workdir is None:
            shutil.rmtree(work, ignore_errors=True)


if __name__ == "__main__":
    main()
