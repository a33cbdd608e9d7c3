"""Item-sharded index generation over the GPUs of one box (one process per GPU, NCCL over NVLink).

The reference's index/ directory is single-process; this is the north-star sharding of
``index/generate_indices.py:85-128``:

* PASS 0 shards naturally - contiguous item blocks per rank, encoder weights and codebooks
  replicated, no communication (the 16 KB/item embeddings never leave their rank);
* collision detection needs a global view, but two items can only ever collide if they share the
  first L-1 codes (the rounds rewrite the LAST level only, generate_indices.py:101-105), so the
  global problem splits into independent PREFIX BUCKETS.  After PASS 0 every item's codes (32 B)
  and residual entering the last level (128 B) travel ONCE, by all-to-all, to the rank that owns its
  bucket (``hash(prefix) % world``); the owner runs the whole <=20-round loop on its buckets locally
  (1/world of the sort and Sinkhorn work, no per-round communication) and a second all-to-all along
  the same routes returns the last-level codes (8 B/item).  Groups, member order and arithmetic are
  exactly those of the single-GPU run, so the result is identical bit for bit.

The arithmetic lives behind a small backend interface so that the host logic above can be
exercised with ``gloo`` on CPU in the tests (where the backend is the numpy oracle); the product
backend is ``CudaBackend`` (C-ABI kernels).  Nothing here falls back to the CPU by itself.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Tuple

import torch
import torch.distributed as dist


@dataclass
class ShardPlan:
    """Contiguous block partition of ``n_total`` items over ``world`` ranks (first ranks get the remainder)."""
    n_total: int
    world: int

    def count(self, rank: int) -> int:
        base, rem = divmod(self.n_total, self.world)
        return base + (1 if rank < rem else 0)

    def start(self, rank: int) -> int:
        base, rem = divmod(self.n_total, self.world)
        return rank * base + min(rank, rem)

    def slice(self, rank: int) -> slice:
        return slice(self.start(rank), self.start(rank) + self.count(rank))

    @property
    def max_count(self) -> int:
        return self.count(0)


def all_gather_rows(local: torch.Tensor, plan: ShardPlan, rank: int, group=None) -> torch.Tensor:
    """Concatenate the ranks' row blocks (ragged blocks are padded to the largest for the collective)."""
    pad = plan.max_count
    buf = local
    if local.shape[0] != pad:
        buf = torch.zeros((pad,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
        buf[: local.shape[0]] = local
    out = torch.empty((plan.world * pad,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, buf.contiguous(), group=group)
    if plan.n_total == plan.world * pad:
        return out
    return torch.cat([out[r * pad: r * pad + plan.count(r)] for r in range(plan.world)], dim=0)


class CudaBackend:
    """Kernels of liblcrec_b200.so on this rank's GPU."""

    def __init__(self, model, n_local_max: int, chunk_rows: int = 131072, n_total: int = None):
        """``n_total``: the rows of the whole job, for ranks that read host blocks (``pass0`` with a layout): the indexer then
        streams in the pieces of the one-GPU run over n_total rows (chunks of min(chunk_rows, n_total) rows)."""
        from . import generate_indices as G
        from . import ops
        self.ops = ops
        self.model = model
        chunk = min(chunk_rows, max(n_local_max if n_total is None else n_total, 1))
        # 5 % slack: the hash-balanced bucket share of a rank may slightly exceed its item share
        self.indexer = G.build_indexer(model, max(int(max(n_local_max, 1) * 1.05) + 1024, chunk), chunk)
        self.cbs = [vq.embedding.weight.detach() for vq in model.rq.vq_layers]
        self.n_codes = [int(c.shape[0]) for c in self.cbs]
        self.eps = float(model.rq.vq_layers[-1].sk_epsilon)
        self.iters = int(model.rq.vq_layers[-1].sk_iters)

    def pass0(self, x_local, n_total: int = None, row_begin: int = 0) -> Tuple[torch.Tensor, torch.Tensor]:
        """Codes + last-level residuals of this rank's shard; an fp16 / bf16 shard is read as it is.  A CUDA tensor goes
        through Indexer.pass0; a host block (CPU tensor or ndarray, e.g. a slice of an ``np.memmap``) is streamed from the
        host as rows [row_begin, row_begin + n) of an ``n_total``-row job (Indexer.pass0_host), so its codes are those of
        the one-GPU run over all n_total rows, bit for bit."""
        n = x_local.shape[0]
        if n == 0:
            dev = self.cbs[0].device
            return (torch.zeros((0, len(self.cbs)), dtype=torch.int64, device=dev),
                    torch.zeros((0, self.cbs[0].shape[1]), dtype=torch.float32, device=dev))
        if isinstance(x_local, torch.Tensor) and x_local.is_cuda:
            self.indexer.pass0(x_local, 0)
        else:
            self.indexer.pass0_host(x_local, n if n_total is None else n_total, row_begin)
        return self.indexer.codes_view(n).clone(), self.indexer.resid_view(n).clone()

    def collisions(self, codes: torch.Tensor) -> dict:
        return self.ops.collisions(codes, self.n_codes)

    def resolve_all(self, resid: torch.Tensor, codes: torch.Tensor, max_rounds: int):
        """All rounds inside the library (lcrec_indexer_resolve); None when the table exceeds the indexer's capacity."""
        if codes.shape[0] > self.indexer.max_items:
            return None
        return self.indexer.resolve_device(codes, resid.contiguous(), max_rounds)

    def resolve(self, resid: torch.Tensor, codes: torch.Tensor, info: dict) -> None:
        flags = self.ops.sinkhorn_groups(resid, self.cbs[-1], info["offsets"], info["members"],
                                         info["counts_dev"][1:2], info["n_groups"], info["n_rows"], self.eps,
                                         self.iters, codes, codes.shape[1] - 1)
        if flags & 6:
            raise RuntimeError(f"sinkhorn_groups failed with flags {flags}")


class NativeExchange:
    """The hand-over of PASS-0 results to the bucket owners and back as native kernels + TWO equal-split all-to-alls
    (csrc/exchange.cu): owner hash + stable partition + record packing in one pass over the items, fixed-size slabs per
    destination (25 % slack over the even share; a header carries the row count), so no split sizes cross the host and the only
    host read is the 8 x 8-byte count vector the owner needs to size its table."""

    def __init__(self, backend, n_local_max: int, world: int, group=None):
        import ctypes as C
        from . import _lib
        self.lib = _lib.load()
        self.C = C
        self.backend, self.world, self.group = backend, int(world), group
        self.L, self.D = len(backend.cbs), int(backend.cbs[0].shape[1])
        self.n_codes = _lib.i32_array(backend.n_codes)
        dev = backend.cbs[0].device
        self.dev = dev
        self.slab_rows = int(n_local_max / world * 1.25) + 4096
        self.slab_bytes = int(self.lib.lcrec_exchange_slab_bytes(self.slab_rows, self.L, self.D))
        self.send = torch.empty(self.slab_bytes * world, dtype=torch.uint8, device=dev)
        self.recv = torch.empty_like(self.send)
        self.back_send = torch.empty((world, self.slab_rows), dtype=torch.int64, device=dev)
        self.back_recv = torch.empty_like(self.back_send)
        self.slot = torch.empty(max(n_local_max, 1), dtype=torch.int32, device=dev)
        self.counts = torch.empty(world, dtype=torch.int64, device=dev)
        self.ws = torch.empty(int(self.lib.lcrec_exchange_workspace_bytes(max(n_local_max, 1), world)), dtype=torch.uint8, device=dev)
        self.cap = world * self.slab_rows
        self.sub_codes = torch.empty((self.cap, self.L), dtype=torch.int64, device=dev)
        self.sub_resid = torch.empty((self.cap, self.D), dtype=torch.float32, device=dev)

    def _st(self):
        return self.C.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)

    def forward(self, codes_local: torch.Tensor, resid_local: torch.Tensor):
        """-> (sub_codes view, sub_resid view) of the rows this rank owns, in ascending global item order; None on EVERY
        rank when a destination slab of ANY rank overflowed (bucket skew beyond the 25 % slack): whether one did is
        all-reduced before the slabs move, so all ranks take the split-size path together and none waits in a collective
        that a failed peer never joins.  Collective."""
        from . import _lib
        from .ops import _p
        n = int(codes_local.shape[0])
        assert n <= self.slot.numel()
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.lcrec_exchange_pack(_p(codes_local), _p(resid_local), n, self.L, self.D, self.n_codes, self.world,
                                                    self.slab_rows, _p(self.send), _p(self.slot), _p(self.counts), _p(self.ws),
                                                    self.ws.numel(), self._st()))
            overflow = (self.counts > self.slab_rows).any().to(torch.int32).view(1)
            dist.all_reduce(overflow, op=dist.ReduceOp.MAX, group=self.group)
            if int(overflow.item()) != 0:
                return None
            dist.all_to_all_single(self.recv, self.send, group=self.group)
            hdr = self.recv.view(self.world, self.slab_bytes)[:, :16].contiguous().view(torch.int64).cpu()
            n_mine = int(hdr[:, 0].sum())
            _lib.check(self.lib.lcrec_exchange_unpack(_p(self.recv), self.world, self.slab_rows, self.L, self.D, _p(self.sub_codes),
                                                      _p(self.sub_resid), n_mine, self._st()))
        return self.sub_codes[:n_mine], self.sub_resid[:n_mine]

    def backward(self, sub_codes: torch.Tensor, codes_local: torch.Tensor) -> torch.Tensor:
        """Resolved last-level codes back to their origin; returns the origin's table (a copy of codes_local, last column updated)."""
        from . import _lib
        from .ops import _p
        out = codes_local.clone()
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.lcrec_exchange_pack_last(_p(sub_codes), self.L, _p(self.recv), self.world, self.slab_rows, self.D,
                                                         _p(self.back_send), int(sub_codes.shape[0]), self._st()))
            dist.all_to_all_single(self.back_recv, self.back_send, group=self.group)
            _lib.check(self.lib.lcrec_exchange_scatter_last(_p(self.back_recv), _p(self.slot), int(out.shape[0]), self.L, _p(out), self._st()))
        return out


def bucket_owner(codes: torch.Tensor, n_codes, world: int) -> torch.Tensor:
    """Owner rank of every item's prefix bucket: the mixed-radix value of the first L-1 codes, mixed with a
    multiplicative hash (so that skewed code usage still spreads evenly), modulo world."""
    prefix = torch.zeros(codes.shape[0], dtype=torch.int64, device=codes.device)
    for l in range(codes.shape[1] - 1):
        prefix = prefix * int(n_codes[l]) + codes[:, l]
    mixed = (prefix * 0x9E3779B97F4A7C15 & 0x7FFFFFFFFFFFFFFF) >> 24      # wraps mod 2^64, then the high bits
    return mixed % world


def resolve_rounds(backend, codes: torch.Tensor, resid: torch.Tensor, max_rounds: int):
    """generate_indices.py:108-128 on one self-contained set of items (codes is updated in place)."""
    n = codes.shape[0]
    if n > 0 and hasattr(backend, "resolve_all"):
        st = backend.resolve_all(resid, codes, max_rounds)
        if st is not None:
            return {k: st[k] for k in ("rounds", "n_unique", "groups_round1", "rows_round1", "sinkhorn_rows", "max_multiplicity")}
    rounds = rows_total = 0
    first = (0, 0)
    info = {"n_unique": n, "max_multiplicity": 1 if n else 0}
    while n > 0:
        info = backend.collisions(codes)
        if rounds == 0:
            first = (info["n_groups"], info["n_rows"])
        if info["n_unique"] == n or rounds >= max_rounds:
            break
        backend.resolve(resid, codes, info)
        rows_total += info["n_rows"]
        rounds += 1
    return {"rounds": rounds, "n_unique": info["n_unique"], "groups_round1": first[0], "rows_round1": first[1],
            "sinkhorn_rows": rows_total, "max_multiplicity": info["max_multiplicity"]}


def generate_codes_sharded(backend, x_local: torch.Tensor, plan: ShardPlan, rank: int, max_rounds: int = 20,
                           group=None, n_codes=None):
    """Sharded ``generate_indices``: returns (codes of this rank's items, stats).  Collective: every
    rank of ``group`` must call it."""
    import os
    on_device = isinstance(x_local, torch.Tensor) and x_local.is_cuda
    timing = os.environ.get("LCREC_DIST_TIMING") == "1" and (on_device or isinstance(backend, CudaBackend))
    marks = []

    def mark(name):
        if timing:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            marks.append((name, e))
    mark("start")
    if not on_device and isinstance(backend, CudaBackend):
        # a host block: streamed in the pieces of the one-GPU run over all plan.n_total rows
        codes_local, resid_local = backend.pass0(x_local, plan.n_total, plan.start(rank))
    else:
        codes_local, resid_local = backend.pass0(x_local)
    mark("pass0")
    n_codes = n_codes or getattr(backend, "n_codes")
    if plan.world == 1:
        codes = codes_local.contiguous()
        stats = resolve_rounds(backend, codes, resid_local, max_rounds)
        stats["collision_rate"] = (plan.n_total - stats["n_unique"]) / max(plan.n_total, 1)
        return codes, stats
    # Every rank sends each item to the owner of its prefix bucket (all-to-all: 160 B/item leave the rank once, instead
    # of every rank gathering all items).  Items arrive grouped by source rank = ascending global item id, because the
    # shards are contiguous blocks and the send order inside a shard is ascending.
    world = plan.world
    last = codes_local.shape[1] - 1
    import os as _os
    if codes_local.is_cuda and hasattr(backend, "indexer") and _os.environ.get("LCREC_EXCHANGE", "native") == "native" and world <= 16:
        ex = getattr(backend, "_native_exchange", None)
        if ex is None or ex.world != world or ex.slot.numel() < codes_local.shape[0] or getattr(backend, "_native_exchange_group", None) is not group:
            ex = backend._native_exchange = NativeExchange(backend, max(plan.max_count, int(codes_local.shape[0])), world, group)
            backend._native_exchange_group = group
        fwd = ex.forward(codes_local.contiguous(), resid_local.contiguous())
    else:
        fwd = None
    if fwd is not None:
        sub_codes, sub_resid = fwd
        mark("partition+exchange")
        st = resolve_rounds(backend, sub_codes, sub_resid, max_rounds)
        mark("rounds")
        out = ex.backward(sub_codes, codes_local)
        n_mine = int(sub_codes.shape[0])
        agg = torch.tensor([st["n_unique"], st["groups_round1"], st["rows_round1"], st["sinkhorn_rows"], st["rounds"], st["max_multiplicity"]],
                           dtype=torch.int64, device=codes_local.device)
        gathered = torch.empty((world, 6), dtype=torch.int64, device=codes_local.device)
        dist.all_gather_into_tensor(gathered, agg.view(1, 6), group=group)         # one collective for all statistics
        gl = gathered.cpu()
        n_unique, g1, r1, rows = [int(v) for v in gl[:, :4].sum(0).tolist()]
        rounds, max_mult = [int(v) for v in gl[:, 4:].max(0).values.tolist()]
        mark("return+stats")
        stats = {"rounds": rounds, "n_unique": n_unique, "groups_round1": g1, "rows_round1": r1, "sinkhorn_rows": rows,
                 "max_multiplicity": max_mult, "collision_rate": (plan.n_total - n_unique) / max(plan.n_total, 1),
                 "bucket_items_this_rank": n_mine}
        if timing:
            stats["timing_ms"] = _report_marks(marks, rank)
        return out, stats
    owner = bucket_owner(codes_local, n_codes, world)
    order = torch.argsort(owner, stable=True)                      # items grouped by destination, ascending inside
    send_counts = torch.bincount(owner, minlength=world)
    recv_counts = torch.empty_like(send_counts)
    dist.all_to_all_single(recv_counts, send_counts, group=group)
    send_splits, recv_splits = send_counts.tolist(), recv_counts.tolist()
    mark("partition+counts")
    n_mine = int(sum(recv_splits))
    sub_codes = torch.empty((n_mine, codes_local.shape[1]), dtype=codes_local.dtype, device=codes_local.device)
    sub_resid = torch.empty((n_mine, resid_local.shape[1]), dtype=resid_local.dtype, device=resid_local.device)
    dist.all_to_all_single(sub_codes, codes_local.index_select(0, order).contiguous(), recv_splits, send_splits, group=group)
    dist.all_to_all_single(sub_resid, resid_local.index_select(0, order).contiguous(), recv_splits, send_splits, group=group)
    mark("exchange")
    st = resolve_rounds(backend, sub_codes, sub_resid, max_rounds)
    mark("rounds")
    # the owners return the resolved last-level codes along the same routes
    back = torch.empty((codes_local.shape[0],), dtype=codes_local.dtype, device=codes_local.device)
    dist.all_to_all_single(back, sub_codes[:, last].contiguous(), send_splits, recv_splits, group=group)
    out = codes_local.clone()
    out[order, last] = back
    agg = torch.tensor([st["n_unique"], st["groups_round1"], st["rows_round1"], st["sinkhorn_rows"]], dtype=torch.int64,
                       device=codes_local.device)
    mx = torch.tensor([st["rounds"], st["max_multiplicity"]], dtype=torch.int64, device=codes_local.device)
    dist.all_reduce(agg, op=dist.ReduceOp.SUM, group=group)
    dist.all_reduce(mx, op=dist.ReduceOp.MAX, group=group)
    n_unique, g1, r1, rows = [int(v) for v in agg.tolist()]
    rounds, max_mult = [int(v) for v in mx.tolist()]
    mark("return+stats")
    stats = {"rounds": rounds, "n_unique": n_unique, "groups_round1": g1, "rows_round1": r1, "sinkhorn_rows": rows,
             "max_multiplicity": max_mult, "collision_rate": (plan.n_total - n_unique) / max(plan.n_total, 1),
             "bucket_items_this_rank": n_mine}
    if timing:
        stats["timing_ms"] = _report_marks(marks, rank)
    return out, stats


def _report_marks(marks, rank: int) -> dict:
    """LCREC_DIST_TIMING=1: ms between consecutive marks of generate_codes_sharded (printed by rank 0 to stderr)."""
    torch.cuda.synchronize()
    ms = {b[0]: a[1].elapsed_time(b[1]) for a, b in zip(marks[:-1], marks[1:])}
    if rank == 0:
        import sys
        print("dist timing (ms): " + ", ".join(f"{k} {v:.2f}" for k, v in ms.items()), file=sys.stderr)
    return ms


# ----------------------------------------------------------------------------------------------------------------
# Data-parallel form of the training-time Sinkhorn (one (global batch x K) problem, rows split over the ranks)
class DistributedSinkhorn:
    """``sinkhorn_algorithm`` (index/models/layers.py:85-108) for a batch whose rows are sharded over the ranks of
    ``group``: the kernel all-reduces the column marginals itself through peer memory (NVLink P2P on symmetric
    buffers, ``lcrec_sinkhorn_dense_dist``) - no collective is launched between iterations.  Reference semantics are
    those of the single-device call on the concatenated batch (SURVEY 8(e)).  Collective: every rank calls it."""

    def __init__(self, n_codes: int, device, group=None):
        import ctypes as C
        import torch.distributed._symmetric_memory as symm
        from . import _lib
        self.lib = _lib.load()
        self.group = group if group is not None else dist.group.WORLD
        self.n_codes = int(n_codes)
        self.device = torch.device(device)
        nbytes = int(self.lib.lcrec_sinkhorn_dist_symmetric_bytes(self.n_codes))
        self.buf = symm.empty(nbytes, dtype=torch.uint8, device=self.device)
        self.buf.zero_()
        self.hdl = symm.rendezvous(self.buf, self.group)
        self.world, self.rank = int(self.hdl.world_size), int(self.hdl.rank)
        self.peers = torch.tensor([int(p) for p in self.hdl.buffer_ptrs], dtype=torch.int64, device=self.device)
        self.epoch = 0
        torch.cuda.synchronize(self.device)
        dist.barrier(group=self.group)          # every buffer is zeroed and mapped before the first kernel polls it

    def center(self, d_local: torch.Tensor) -> torch.Tensor:
        """center_distance_for_constraint (vq.py:51-61) with the max / min taken over the GLOBAL batch."""
        mm = torch.stack([d_local.max(), -d_local.min()]) if d_local.numel() else torch.full((2,), -float("inf"), device=self.device)
        dist.all_reduce(mm, op=dist.ReduceOp.MAX, group=self.group)
        mx, mn = mm[0], -mm[1]
        mid = (mx + mn) / 2
        amp = mx - mid + 1e-5
        return (d_local - mid) / amp

    def __call__(self, distances_local: torch.Tensor, epsilon: float, iters: int, n_rows_global: int = None):
        import ctypes as C
        from . import _lib
        from .ops import _p, _stream, _ws
        d = distances_local.detach().to(torch.float64).contiguous()
        b, k = d.shape
        assert k == self.n_codes and d.is_cuda
        if n_rows_global is None and getattr(self, "n_rows_hint", None) is not None:
            n_rows_global = int(self.n_rows_hint)       # set by a caller that knows the global batch (no host read)
        if n_rows_global is None:
            t = torch.tensor([b], dtype=torch.int64, device=self.device)
            dist.all_reduce(t, group=self.group)
            n_rows_global = int(t.item())
        q = torch.empty_like(d)
        arg = torch.empty((b,), dtype=torch.int64, device=self.device)
        flags = torch.zeros(1, dtype=torch.int32, device=self.device)
        ws = _ws(self.lib.lcrec_sinkhorn_workspace_bytes(max(b, 1), k), self.device)
        epoch = self.epoch
        self.epoch += int(iters) + 1            # exactly the steps this call publishes: slots alternate across calls
        with torch.cuda.device(self.device):
            _lib.check(self.lib.lcrec_sinkhorn_dense_dist(_p(d), b, int(n_rows_global), k, float(epsilon), int(iters), _p(q), _p(arg),
                                                          _p(flags), _p(self.peers), self.world, self.rank, C.c_uint64(epoch),
                                                          _p(ws), ws.numel(), _stream(d)))
        return q, arg, flags


# ----------------------------------------------------------------------------------------------------------------
# Data-parallel form of the EMA codebook step of index_improve (one step over the global batch, rows split over the ranks)
class DistributedEma:
    """The EMA step of index_improve's VectorQuantizer (``lcrec_ema_update``) for a batch whose rows are split over the
    ranks of ``group`` in ``ShardPlan`` blocks.  Each call gathers every rank's (latent, indices) block through peer memory
    (symmetric buffers, ``lcrec_ema_update_dist``) and runs the single-device kernel on the concatenated batch, so the
    buffers end bit-identical to the single-device step on the global batch, on every rank.  One instance serves every
    level of a model: ``rows_per_rank`` (the largest block, ``ShardPlan(batch_size, world).max_count``) and ``e_dim`` fix
    the buffer layout; the number of codes and the rows of a call may vary.  Collective: every rank calls ``update``."""

    def __init__(self, rows_per_rank: int, e_dim: int, device, group=None):
        import torch.distributed._symmetric_memory as symm
        from . import _lib
        self.lib = _lib.load()
        self.group = group if group is not None else dist.group.WORLD
        self.rows_per_rank, self.e_dim = int(rows_per_rank), int(e_dim)
        self.device = torch.device(device)
        nbytes = int(self.lib.lcrec_ema_dist_symmetric_bytes(self.rows_per_rank, self.e_dim))
        if nbytes <= 0:
            raise ValueError(f"DistributedEma: rows_per_rank {rows_per_rank} and e_dim {e_dim} must be >= 1")
        self.buf = symm.empty(nbytes, dtype=torch.uint8, device=self.device)
        self.buf.zero_()
        self.hdl = symm.rendezvous(self.buf, self.group)
        self.world, self.rank = int(self.hdl.world_size), int(self.hdl.rank)
        self.peers = torch.tensor([int(p) for p in self.hdl.buffer_ptrs], dtype=torch.int64, device=self.device)
        cap = self.world * self.rows_per_rank
        self.gathered_latent = torch.empty((cap, self.e_dim), dtype=torch.float32, device=self.device)
        self.gathered_indices = torch.empty((cap,), dtype=torch.int64, device=self.device)
        self.epoch = 0                          # calls made on the buffers: the publish counters only grow
        self.n_rows_hint = None                 # the global row count of the current batch, set by a caller that knows it
        torch.cuda.synchronize(self.device)
        dist.barrier(group=self.group)          # every buffer is zeroed and mapped before the first kernel polls it

    def update(self, latent_local: torch.Tensor, indices_local: torch.Tensor, n_global, cluster_size: torch.Tensor,
               ema_w: torch.Tensor, codebook: torch.Tensor, decay: float, eps: float) -> torch.Tensor:
        """The EMA step in place on (cluster_size, ema_w, codebook); returns the gathered global latent (n_global, e_dim), a
        view that the next call overwrites.  ``n_global`` None: ``n_rows_hint``, else an all-reduce of the block sizes."""
        import ctypes as C
        from . import _lib
        from .ops import _inplace_f32, _need_cuda, _p, _stream, check_later
        _need_cuda(latent_local, indices_local, cluster_size, ema_w, codebook)
        k, d = codebook.shape
        if d != self.e_dim:
            raise ValueError(f"DistributedEma: codebook e_dim {d}, buffers laid out for {self.e_dim}")
        lat = latent_local.detach().reshape(-1, d).to(torch.float32).contiguous()
        idx = indices_local.detach().reshape(-1).to(torch.int64).contiguous()
        n = int(lat.shape[0])
        if idx.shape[0] != n:
            raise ValueError("DistributedEma: one index per latent row expected")
        if n_global is None:
            n_global = self.n_rows_hint
        if n_global is None:
            t = torch.tensor([n], dtype=torch.int64, device=self.device)
            dist.all_reduce(t, group=self.group)
            n_global = int(t.item())
        n_global = int(n_global)
        plan = ShardPlan(n_global, self.world)
        # decided from the global row count, which every rank shares: an oversized batch raises on every rank
        if plan.max_count > self.rows_per_rank:
            raise ValueError(f"DistributedEma: a block of {plan.max_count} rows exceeds rows_per_rank = {self.rows_per_rank}")
        # a block other than this rank's ShardPlan share would gather rows the peers never published; raise before any
        # device work (the peers, if their blocks are right, see this rank's absence through the bounded wait's flag)
        if n != plan.count(self.rank):
            raise ValueError(f"DistributedEma: rank {self.rank} holds {n} rows, its ShardPlan share of {n_global} is "
                             f"{plan.count(self.rank)}")
        _inplace_f32(cluster_size, "cluster_size"); _inplace_f32(ema_w, "ema_w"); _inplace_f32(codebook, "codebook")
        flags = torch.empty(1, dtype=torch.int32, device=self.device)
        epoch = self.epoch
        self.epoch += 1
        with torch.cuda.device(self.device):
            _lib.check(self.lib.lcrec_ema_update_dist(_p(lat), _p(idx), n, n_global, k, d, float(decay), float(eps),
                                                      _p(cluster_size), _p(ema_w), _p(codebook), _p(self.gathered_latent),
                                                      _p(self.gathered_indices), _p(flags), _p(self.peers), self.world,
                                                      self.rank, self.rows_per_rank, C.c_uint64(epoch), _stream(lat)))
        check_later("ema_dist", flags)
        return self.gathered_latent[:n_global]
