"""Data-parallel training of the RQ-VAE over the GPUs of one box (SURVEY 8(e), "Training DP").

The reference's ``index/trainer.py`` is single-device; the parity target is therefore the single-device step on the GLOBAL
batch.  One process per GPU (``torch.distributed``, NCCL over NVLink), model replicated, every rank reads the same global
batches (same loader, same shuffle seed) and takes a contiguous row block of each (``ShardPlan``).  Per step, these
things cross NVLink:

* the Sinkhorn level is ONE (global batch x K) problem (``vq.py:77-79``): ``DistributedSinkhorn`` keeps the row steps local
  and all-reduces the column marginals inside the kernel through peer memory (plus one 2-element MAX all-reduce for the
  centring of ``vq.py:54-55``);
* the gradients: every loss of the step is a mean over batch rows, so rank r back-propagates ``loss_r * n_r / N`` and
  ``all_reduce(SUM)`` over a flat buffer that holds every gradient (encoder + decoder 89.5 MB, codebooks 128 KB) yields the
  gradient of the global-batch loss on every rank - in ~32 MB buckets that start as soon as autograd has produced their
  gradients (decoder first), overlapping the rest of the backward pass; clipping and the optimiser step then run identically everywhere
  (``lcrec_adam_clip_step``), so the replicas never diverge;
* for index_improve's EMA-codebook model, per level the row block of the latent and its codes: ``DistributedEma`` gathers
  every rank's block through peer memory and runs the single-device EMA kernel on the global batch, so counts, sums and
  codebooks are bit-identical to the single-device step and equal on every rank.  A dead-code reset (every
  ``reset_interval`` steps, decided from the shared counts) is drawn by rank 0 on the gathered latent and broadcast.

Codebook k-means initialisation (first batch, ``vq.py:67-68``) runs on the full global batch on every rank with the same
numpy seed, after which rank 0's codebooks are broadcast.  BatchNorm in training mode runs SYNCHRONISED: its kernels all-reduce the
per-channel sums of the forward and of the backward pass over the ranks (global-batch statistics, identical running
statistics everywhere).  The k-means pass of an EMA model takes no EMA step (the first batch gets one, in the training
forward).  A rank whose row block is empty still joins the Sinkhorn and EMA collectives.  Rank 0 writes checkpoints.
"""
from __future__ import annotations

import torch
import torch.distributed as dist
from tqdm import tqdm

from . import ops
from .distributed import ShardPlan
from .optim import FusedAdam
from .trainer import Trainer
from .utils import set_color


class DataParallelTrainer(Trainer):
    def __init__(self, args, model, data_num, group=None):
        if not dist.is_initialized():
            raise RuntimeError("DataParallelTrainer needs an initialised torch.distributed process group")
        self.group = group if group is not None else dist.group.WORLD
        self.rank = dist.get_rank(self.group)
        self.world = dist.get_world_size(self.group)
        # BatchNorm (what `run.sh --bn False` really trains, main.py:31): the single-device semantics need batch statistics
        # over the GLOBAL batch -> the BN kernels all-reduce their per-channel sums over the group (forward and backward)
        self._bn_modules = [m for m in model.modules() if isinstance(m, torch.nn.modules.batchnorm._BatchNorm)]
        super().__init__(args, model, data_num)
        self._flat = None
        self._flat_params = None
        self._sinkhorn_levels = []
        self._ema = None
        for p in self.model.parameters():                       # identical replicas whatever the local seed was
            dist.broadcast(p.data, src=dist.get_global_rank(self.group, 0) if self.group is not dist.group.WORLD else 0,
                           group=self.group)
        if self.device.type == "cuda":
            self._hook_distributed_sinkhorn()
            self._hook_distributed_ema()

    # ---- the Sinkhorn level as one global problem
    def _hook_distributed_sinkhorn(self):
        from .distributed import DistributedSinkhorn
        rq = getattr(self.model, "rq", None)
        for q in (rq.vq_layers if rq is not None else []):
            if getattr(q, "sk_epsilon", 0) and q.sk_epsilon > 0:
                if getattr(q, "dist_sinkhorn", None) is None:
                    q.dist_sinkhorn = DistributedSinkhorn(q.n_e, self.device, self.group)
                self._sinkhorn_levels.append(q)

    # ---- index_improve's EMA codebooks: one EMA step over the global batch
    def _ema_levels(self):
        rq = getattr(self.model, "rq", None)
        return [q for q in (rq.vq_layers if rq is not None else []) if hasattr(q, "_ema_cluster_size")]

    def _hook_distributed_ema(self):
        """One DistributedEma serves every EMA level (the levels run one after the other on the same stream), sized for the
        largest row block of a batch of args.batch_size rows.  The EMA buffers are broadcast like the parameters."""
        from .distributed import DistributedEma
        levels = self._ema_levels()
        if not levels:
            return
        self._ema = DistributedEma(ShardPlan(int(self.args.batch_size), self.world).max_count, levels[0].e_dim, self.device,
                                   self.group)
        src = dist.get_global_rank(self.group, 0) if self.group is not dist.group.WORLD else 0
        for q in levels:
            q.dist_ema = self._ema
            for t in (q._ema_cluster_size, q._ema_w):
                dist.broadcast(t, src=src, group=self.group)

    # ---- gradient reduction: flat buffer, buckets reduced WHILE the backward pass is still running
    BUCKET_ELEMS = 8 * 1024 * 1024        # ~32 MB of fp32 per all-reduce: the decoder's last layer alone, then groups of smaller layers

    def _setup_buckets(self):
        """One flat fp32 buffer holds every gradient (parameter order); it is cut into buckets of consecutive parameters in the
        order autograd produces them (REVERSE parameter order: decoder first).  A post-accumulate-grad hook copies each gradient
        into its slot; when a bucket is complete its all-reduce starts asynchronously - on NCCL's stream, overlapping the rest of
        the backward pass - strictly in bucket order on every rank, so that the collectives line up even when a rank has no rows
        and issues them all at the end."""
        params = [p for p in self.model.parameters() if p.requires_grad]
        self._params = params
        total = sum(p.numel() for p in params)
        self._flat = torch.zeros(total, dtype=torch.float32, device=self.device)
        self._views, off = [], 0
        offs = []
        for p in params:
            offs.append(off)
            self._views.append(self._flat[off: off + p.numel()].view_as(p))
            off += p.numel()
        self._buckets = []                 # (first param index, last param index) in issue order
        hi = len(params) - 1
        while hi >= 0:
            lo, size = hi, params[hi].numel()
            while lo > 0 and size + params[lo - 1].numel() <= self.BUCKET_ELEMS:
                lo -= 1
                size += params[lo].numel()
            self._buckets.append((lo, hi))
            hi = lo - 1
        self._bucket_of = {}
        for b, (lo, hi) in enumerate(self._buckets):
            for i in range(lo, hi + 1):
                self._bucket_of[i] = b
        self._offs = offs
        self._index = {id(p): i for i, p in enumerate(params)}
        for p in params:
            p.register_post_accumulate_grad_hook(self._on_grad)
        self._reset_reduce()

    def _reset_reduce(self):
        self._pending = [hi - lo + 1 for lo, hi in self._buckets]
        self._have = [False] * len(self._params)
        self._handles = []
        self._next_bucket = 0
        self._reducing = False

    def _bucket_slice(self, b):
        lo, hi = self._buckets[b]
        return self._flat[self._offs[lo]: self._offs[hi] + self._params[hi].numel()]

    def _issue_ready(self):
        while self._next_bucket < len(self._buckets) and self._pending[self._next_bucket] == 0:
            self._handles.append(dist.all_reduce(self._bucket_slice(self._next_bucket), op=dist.ReduceOp.SUM, group=self.group, async_op=True))
            self._next_bucket += 1

    def _on_grad(self, p):
        if not self._reducing:
            return                                               # (a backward outside the training step, e.g. a user's probe)
        i = self._index[id(p)]
        if self._have[i]:
            return
        self._views[i].copy_(p.grad)
        self._have[i] = True
        self._pending[self._bucket_of[i]] -= 1
        self._issue_ready()

    def _all_reduce_grads(self):
        """Finish the step's reduction: parameters that produced no gradient (a rank without rows, an unused parameter) contribute
        zeros, the remaining buckets are issued in order, and every gradient then lives in the flat buffer (no copy back)."""
        if getattr(self, "_params", None) is None:
            self._setup_buckets()
            self._reducing = True
            for i, p in enumerate(self._params):                 # the hooks were registered after this step's backward
                if p.grad is not None:
                    self._on_grad(p)
        for i, have in enumerate(self._have):
            if not have:
                self._views[i].zero_()
                self._have[i] = True
                self._pending[self._bucket_of[i]] -= 1
        self._issue_ready()
        for h in self._handles:
            h.wait()
        for p, v in zip(self._params, self._views):
            p.grad = v
        self._reset_reduce()

    def _init_codebooks_on_global_batch(self, data):
        """First training batch (vq.py:67-68): every level's k-means runs on the FULL global batch, on every rank, with the
        caller's `use_sk` - in the reference's single-device step the residual that feeds level l + 1's k-means comes from
        level l's Sinkhorn assignment whenever that level has sk_epsilon > 0.  Every rank holds all the rows here, so the
        Sinkhorn levels use the local dense kernel for this one pass.  Afterwards the codebooks are broadcast from rank 0:
        replica equality must not rest on every rank's numpy RNG being in the same state."""
        rq = getattr(self.model, "rq", None)
        if rq is None or not any(not q.initted for q in rq.vq_layers):
            return
        saved = [(q, q.dist_sinkhorn) for q in rq.vq_layers if getattr(q, "dist_sinkhorn", None) is not None]
        for q, _ in saved:
            q.dist_sinkhorn = None
        bn_saved = [(bn, getattr(bn, "lcrec_sync", None), {k: v.clone() for k, v in bn.state_dict().items() if "running" in k or "tracked" in k})
                    for bn in getattr(self, "_bn_modules", [])]
        for bn, _, _ in bn_saved:
            bn.lcrec_sync = None                                # the full batch is local in this pass
        # an EMA model takes no EMA step in this pass: the first batch gets exactly one, in the training forward
        kw = {"use_ema": False} if self._ema_levels() else {}
        try:
            with torch.no_grad():
                self.model(data.to(self.device), **kw)
        finally:
            for q, ds in saved:
                q.dist_sinkhorn = ds
            for bn, sync, bufs in bn_saved:                     # this extra forward must not count as a training step of the BN layers
                bn.lcrec_sync = sync
                for k, v in bufs.items():
                    getattr(bn, k).copy_(v)
        src = dist.get_global_rank(self.group, 0) if self.group is not dist.group.WORLD else 0
        for q in rq.vq_layers:
            if hasattr(q, "embedding"):
                dist.broadcast(q.embedding.weight.data, src=src, group=self.group)

    def _join_forward_collectives(self):
        """A rank whose row block of this batch is empty still has to take part in the collectives of the forward pass, in
        the forward's level order: per Sinkhorn level the 2-element MAX all-reduce of the centring and the in-kernel arrival
        of the marginal all-reduce, per EMA level the EMA step with 0 local rows (and the reset broadcast when it is due).
        Skipping them would leave the peers' collectives mismatched with this rank's next one."""
        rq = getattr(self.model, "rq", None)
        for q in (rq.vq_layers if rq is not None else []):
            if q in self._sinkhorn_levels:
                d = torch.empty((0, q.n_e), dtype=torch.float32, device=self.device)
                dc = q.dist_sinkhorn.center(d)
                _, _, flags = q.dist_sinkhorn(dc, q.sk_epsilon, q.sk_iters)
                ops.check_later("sinkhorn", flags)
            if getattr(q, "dist_ema", None) is not None:
                q.ema_step(torch.empty((0, q.e_dim), dtype=torch.float32, device=self.device),
                           torch.empty((0,), dtype=torch.int64, device=self.device))

    def _train_epoch(self, train_data, epoch_idx):
        self.model.train()
        total_loss = 0
        total_recon_loss = 0
        bar = tqdm(train_data, total=len(train_data), ncols=100, desc=set_color(f"Train {epoch_idx}", "pink"),
                   disable=self.rank != 0)
        for data in bar:
            n = data.shape[0]
            plan = ShardPlan(n, self.world)
            local = data[plan.slice(self.rank)].to(self.device)
            weight = local.shape[0] / max(n, 1)
            for q in self._sinkhorn_levels:
                q.dist_sinkhorn.n_rows_hint = n                 # the global row count, known here: no all-reduce + host read
            if self._ema is not None:
                self._ema.n_rows_hint = n
            if self._bn_modules:
                if n < self.world:
                    raise RuntimeError(f"synchronised BatchNorm: a batch of {n} rows leaves a rank of {self.world} without rows")
                for bn in self._bn_modules:
                    bn.lcrec_sync = (self.group, n) if self.device.type == "cuda" else None
            with ops.defer_checks():
                self.optimizer.zero_grad()
                self._reducing = getattr(self, "_params", None) is not None      # hooks copy + reduce during this step's backward
                self._init_codebooks_on_global_batch(data)
                stats = torch.zeros(2, dtype=torch.float32, device=self.device)
                if local.shape[0] > 0:
                    out, rq_loss, _ = self._model_forward(local)
                    loss, loss_recon = self.model.compute_loss(out, rq_loss, xs=local)
                    (loss * weight).backward()
                    stats = torch.stack([loss.detach(), loss_recon.detach()]).float() * weight
                else:
                    self._join_forward_collectives()
                self._all_reduce_grads()
                dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=self.group)     # the global-batch loss values
                self._check_nan(stats[0])
                if isinstance(self.optimizer, FusedAdam) or hasattr(self.optimizer, "clip_and_step"):
                    self.optimizer.clip_and_step(1.0)
                else:
                    torch.nn.utils.clip_grad_norm_(self.model.parameters(), 1.0)
                    self.optimizer.step()
                self.scheduler.step()
                total_loss += stats[0].item()
                total_recon_loss += stats[1].item()
        return total_loss, total_recon_loss

    def _save_checkpoint(self, epoch, collision_rate=1, ckpt_file=None):
        if self.rank != 0:
            import os
            name = ckpt_file if ckpt_file else "epoch_%d_collision_%.4f_model.pth" % (epoch, collision_rate)
            return os.path.join(self.ckpt_dir, name)
        return super()._save_checkpoint(epoch, collision_rate=collision_rate, ckpt_file=ckpt_file)
