"""Index generation with collision resolution - the north-star path.

Function + CLI equivalent of the flat reference script ``index/generate_indices.py`` (:44-145):
load a checkpoint, PASS 0 argmin codes for every item, force ``sk_epsilon`` = 0 on levels 0..L-2
and 0.003 on the last level if it was 0 (:101-105), then up to 20 rounds in which every group of
items sharing a code tuple is re-quantised ON ITS OWN with Sinkhorn on the last level (:107-128),
finally ``{item: ["<a_i>", "<b_j>", ...]}`` as JSON (:138-145).

All of the arithmetic (encoder GEMMs, residual quantisation, sort/unique grouping, per-group
Sinkhorn) runs in liblcrec_b200.so behind ``lcrec_indexer_*``; nothing is computed on the CPU.
The reference's hard-coded ``dataset / ckpt_path / output_dir / device`` lines are CLI flags here.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time
from typing import Optional

import numpy as np
import torch

from . import ops
from .datasets import EmbDataset
from .models.rqvae import RQVAE

PREFIX = ["<a_{}>", "<b_{}>", "<c_{}>", "<d_{}>", "<e_{}>"]       # generate_indices.py:83


def apply_generation_epsilons(model: RQVAE) -> float:
    """generate_indices.py:101-105 (mutates the model exactly like the script)."""
    for vq in model.rq.vq_layers[:-1]:
        vq.sk_epsilon = 0.0
    last = model.rq.vq_layers[-1]
    if last.sk_epsilon == 0.0:
        last.sk_epsilon = 0.003
    return float(last.sk_epsilon)


def build_indexer(model: RQVAE, max_items: int, chunk_rows: int = 131072) -> ops.Indexer:
    model.eval()
    eps = apply_generation_epsilons(model)
    with torch.no_grad():
        if not model.encoder._fused_ok():
            raise RuntimeError("encoder must be a ReLU MLP in eval mode for index generation")
        handle = model.encoder._get_handle()
    cbs = [vq.embedding.weight.detach() for vq in model.rq.vq_layers]
    return ops.Indexer(handle, cbs, eps, model.rq.vq_layers[-1].sk_iters, max_items, chunk_rows)


@torch.no_grad()
def generate_codes(model: RQVAE, data, max_rounds: int = 20, chunk_rows: int = 131072, indexer=None):
    """Collision-resolved codes for every row of ``data``.

    ``data``: CUDA float tensor (device-resident path) or CPU tensor / ndarray / EmbDataset (host
    path: embeddings are streamed to the device in chunks).  fp16 / bf16 embeddings are indexed as they are
    (an fp16 ndarray or ``.npy`` is not converted; the codes equal those of its fp32 upcast); other ndarray
    dtypes become an fp32 copy.  Returns (codes int64 CPU tensor, stats).
    """
    if isinstance(data, EmbDataset):
        data = data.embeddings
    if isinstance(data, np.ndarray):
        data = torch.from_numpy(np.ascontiguousarray(data, dtype=np.float16 if data.dtype == np.float16 else np.float32))
    n = int(data.shape[0])
    ix = indexer or build_indexer(model, max(n, 1), min(chunk_rows, max(n, 1)))
    if data.is_cuda:
        codes, stats = ix.run_device(data, max_rounds)
        codes = codes.cpu()
    else:
        codes, stats = ix.run_host(data.contiguous(), max_rounds=max_rounds)
    stats["collision_rate"] = (n - stats["n_unique"]) / max(n, 1)
    return codes, stats


def codes_to_index_dict(codes) -> dict:
    arr = np.asarray(codes)
    return {item: [PREFIX[i].format(int(v)) for i, v in enumerate(row)] for item, row in enumerate(arr.tolist())}


def write_index_json(codes, output_file: str) -> None:
    """generate_indices.py:138-145.  A CUDA code table is formatted on the device (``ops.index_json_bytes``: the same bytes,
    ~ms at 1 M items instead of seconds of Python); a host array goes through the reference's own dict + json.dump."""
    if isinstance(codes, torch.Tensor) and codes.is_cuda:
        with open(output_file, "wb") as fp:
            fp.write(ops.index_json_bytes(codes))
        return
    with open(output_file, "w") as fp:
        json.dump(codes_to_index_dict(codes), fp)                  # generate_indices.py:144-145


def write_index_json_parts(fragment: bytes, output_file: str, group=None) -> None:
    """Collective: the `.index.json` of a table whose row blocks are spread over the ranks of ``group`` in rank order, from
    each rank's fragment (``ops.index_json_bytes(codes, item_base, braces=False)``).  One all-gather of the fragment lengths
    gives every rank its byte offset; rank 0 creates the file at its final size and writes the braces, then every rank
    writes its bytes in place with one positional write (the ranks share one host's file system)."""
    import torch.distributed as dist
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend(group) == "nccl" else torch.device("cpu")
    lens = torch.empty(world, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(lens, torch.tensor([len(fragment)], dtype=torch.int64, device=dev), group=group)
    lens = lens.tolist()
    total = 2 + sum(lens)
    if rank == 0:
        fd = os.open(output_file, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o666)
        try:
            os.ftruncate(fd, total)
            os.pwrite(fd, b"{", 0)
            os.pwrite(fd, b"}", total - 1)
        finally:
            os.close(fd)
    dist.barrier(group=group)                                  # the file exists at its size before anyone writes into it
    if fragment:
        fd = os.open(output_file, os.O_WRONLY)
        try:
            view, off = memoryview(fragment), 1 + sum(lens[:rank])
            while view:                                         # pwrite may write less than asked
                k = os.pwrite(fd, view, off)
                view, off = view[k:], off + k
        finally:
            os.close(fd)
    dist.barrier(group=group)                                  # the file is complete when any rank returns


def load_model(ckpt_path: str, device, in_dim: Optional[int] = None, data_path: Optional[str] = None, mmap: bool = False):
    """generate_indices.py:51-74 (``weights_only=False``: the checkpoint pickles an argparse.Namespace).  ``mmap``: the
    embeddings are a read-only memory map of the ``.npy`` instead of a copy in host memory."""
    ckpt = torch.load(ckpt_path, map_location=torch.device("cpu"), weights_only=False)
    args = ckpt["args"]
    data = EmbDataset(data_path or args.data_path, mmap=mmap)
    model = RQVAE(in_dim=in_dim or data.dim, num_emb_list=args.num_emb_list, e_dim=args.e_dim, layers=args.layers,
                  dropout_prob=args.dropout_prob, bn=args.bn, loss_type=args.loss_type,
                  quant_loss_weight=args.quant_loss_weight, kmeans_init=args.kmeans_init,
                  kmeans_iters=args.kmeans_iters, sk_epsilons=args.sk_epsilons, sk_iters=args.sk_iters)
    model.load_state_dict(ckpt["state_dict"])
    return model.to(device).eval(), data, args


def main(argv=None):
    ap = argparse.ArgumentParser(description="LC-Rec index generation (B200)")
    ap.add_argument("--dataset", default="Games")
    ap.add_argument("--ckpt_path", required=True)
    ap.add_argument("--output_dir", required=True)
    ap.add_argument("--data_path", default=None, help="override args.data_path stored in the checkpoint")
    ap.add_argument("--device", default="cuda:0")
    ap.add_argument("--max_rounds", type=int, default=20)
    ap.add_argument("--chunk_rows", type=int, default=131072)
    ap.add_argument("--dist_timeout", type=float, default=1800.0,
                    help="seconds a rank waits in a collective before it fails (under torchrun)")
    a = ap.parse_args(argv)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        return _main_sharded(a, world)
    device = torch.device(a.device)
    timing = os.environ.get("LCREC_DIST_TIMING") == "1"
    t0 = time.perf_counter()
    model, data, _ = load_model(a.ckpt_path, device, data_path=a.data_path)
    print(model)
    t1 = time.perf_counter()
    if timing:
        ops.profile_enable(True)                                   # stage events: the rounds apart from PASS 0
    codes, stats = generate_codes(model, data, a.max_rounds, a.chunk_rows)
    t2 = time.perf_counter()
    print("All indices number: ", len(codes))
    print("Max number of conflicts: ", stats["max_multiplicity"])
    print("Collision Rate", stats["collision_rate"])
    os.makedirs(a.output_dir, exist_ok=True)
    out = os.path.join(a.output_dir, f"{a.dataset}.index.json")
    if not timing:
        write_index_json(codes.to(device), out)                    # formatted on the device
        return out
    text = ops.index_json_bytes(codes.to(device))                  # what write_index_json does, timed in two parts
    t3 = time.perf_counter()
    with open(out, "wb") as fp:
        fp.write(text)
    t4 = time.perf_counter()
    prof = ops.profile_collect()
    ops.profile_enable(False)
    rounds_s = sum(ms for tag, (ms, _) in prof.items() if 21 <= tag <= 26) / 1e3      # collision checks + Sinkhorn (GPU time)
    phases = {"setup_s": t1 - t0, "codes_s": t2 - t1, "pass0_streaming_s": t2 - t1 - rounds_s, "rounds_s": rounds_s,
              "json_s": t3 - t2, "write_s": t4 - t3}
    print("generate timing: " + json.dumps(phases), file=sys.stderr)
    return out


def _main_sharded(a, world: int) -> str:
    """``main`` under torchrun: one process per GPU of the box.  Rank r streams its ShardPlan block of the memory-mapped
    embeddings from the host (in the pieces of the one-GPU run, so PASS 0 gives the same codes), the prefix buckets are
    exchanged and resolved by their owners (distributed.generate_codes_sharded), and every rank writes its part of the JSON
    at its offset.  The file and the printed lines are those of the one-GPU run, byte for byte."""
    import datetime
    import torch.distributed as dist
    from .distributed import CudaBackend, ShardPlan, generate_codes_sharded
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device(f"cuda:{local_rank}")
    dist.init_process_group("nccl", timeout=datetime.timedelta(seconds=a.dist_timeout))
    try:
        rank = dist.get_rank()
        timing = os.environ.get("LCREC_DIST_TIMING") == "1"
        t0 = time.perf_counter()
        model, data, _ = load_model(a.ckpt_path, device, data_path=a.data_path, mmap=True)
        if rank == 0:
            print(model)
        x = data.embeddings
        n = int(x.shape[0])
        plan = ShardPlan(n, world)
        backend = CudaBackend(model, plan.max_count, a.chunk_rows, n_total=n)
        t1 = time.perf_counter()
        codes, stats = generate_codes_sharded(backend, x[plan.slice(rank)], plan, rank, a.max_rounds)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        if rank == 0:
            print("All indices number: ", n)
            print("Max number of conflicts: ", stats["max_multiplicity"])
            print("Collision Rate", stats["collision_rate"])
            os.makedirs(a.output_dir, exist_ok=True)
        out = os.path.join(a.output_dir, f"{a.dataset}.index.json")
        fragment = ops.index_json_bytes(codes, item_base=plan.start(rank), braces=False)      # formatted on this rank's device
        t3 = time.perf_counter()
        write_index_json_parts(fragment, out)
        t4 = time.perf_counter()
        if timing and rank == 0:
            phases = {"setup_s": t1 - t0, "codes_s": t2 - t1, "json_s": t3 - t2, "write_s": t4 - t3}
            phases.update({f"{k}_ms": v for k, v in stats.get("timing_ms", {}).items()})
            print("generate timing: " + json.dumps(phases), file=sys.stderr)
        return out
    finally:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
