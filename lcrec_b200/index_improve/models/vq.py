"""One codebook level with EMA update, dead-code reset and usage statistics.
Import surface of reference ``index_improve/models/vq.py`` (VectorQuantizer :7-217): same constructor, buffers
(``_ema_cluster_size``, ``_ema_w`` - state_dict compatible), ``forward(x, use_sk=True, use_ema=True)``,
``get_codebook_usage()``.  Index selection is the base class's (argmin / Sinkhorn kernels); the EMA block :146-187 is ONE
kernel (``lcrec_ema_update``: per-code sums in item order, bit-identical to the CPU ``index_add_``), the usage statistic
another.  The reset (:79-114) keeps the reference's sequence of torch RNG draws (randint, randperm, randn_like on the
latent's device), so a reference run on the same device with the same seed resets the same codes to the same vectors.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from ... import ops
from ...models.vq import VectorQuantizer as _BaseVectorQuantizer


class VectorQuantizer(_BaseVectorQuantizer):
    def __init__(self, n_e, e_dim, beta=0.25, kmeans_init=False, kmeans_iters=10, sk_epsilon=0.003, sk_iters=100,
                 ema_decay=0.99, epsilon=1e-5, reset_threshold=1e-5, reset_interval=1000):
        super().__init__(n_e, e_dim, beta=beta, kmeans_init=kmeans_init, kmeans_iters=kmeans_iters,
                         sk_epsilon=sk_epsilon, sk_iters=sk_iters)
        self.ema_decay = ema_decay
        self.epsilon = epsilon
        self.reset_threshold = reset_threshold
        self.reset_interval = reset_interval
        self.step_count = 0
        self.register_buffer("_ema_cluster_size", torch.zeros(n_e))
        self.register_buffer("_ema_w", torch.zeros(n_e, e_dim))
        # data-parallel training: a lcrec_b200.distributed.DistributedEma makes the EMA step ONE step over the global batch
        # (the ranks' row blocks gathered through peer memory, identical buffers on every rank); None = local
        self.dist_ema = None

    @torch.no_grad()
    def _reset_unused_codes(self, latent):
        """vq.py:79-114.  The dead-code mask comes from the usage kernel; one host read (the count) like the reference's
        ``.item()``; the draws and the three scattered writes are torch calls in the reference's order."""
        _, unused_mask = ops.codebook_usage(self._ema_cluster_size, self.epsilon, self.reset_threshold, want_unused=True)
        num_unused = int(unused_mask.sum().item())
        if num_unused == 0 or len(latent) == 0:
            return
        unused_indices = torch.where(unused_mask)[0]
        num_samples = min(num_unused, len(latent))
        sample_indices = torch.randint(0, len(latent), (num_samples,), device=latent.device)
        sample_vectors = latent[sample_indices]
        if num_unused > num_samples:
            selected = unused_indices[torch.randperm(len(unused_indices), device=latent.device)[:num_samples]]
        else:
            selected = unused_indices
        noise = torch.randn_like(sample_vectors) * 0.01
        self.embedding.weight.data[selected] = (sample_vectors + noise).detach()
        self._ema_cluster_size[selected] = 0
        self._ema_w[selected] = 0

    def forward(self, x, use_sk=True, use_ema=True):
        latent = x.view(-1, self.e_dim)
        if not self.initted and self.training:
            self.init_emb(latent)
        indices = self.assign(latent.detach(), use_sk)
        x_q = self.embedding(indices).view(x.shape)
        commitment_loss = F.mse_loss(x_q.detach(), x)
        codebook_loss = F.mse_loss(x_q, x.detach())
        loss = codebook_loss + self.beta * commitment_loss
        x_q = x + (x_q - x).detach()                  # forward value uses the codebook BEFORE the EMA step (vq.py:138,198)
        if self.training and use_ema:
            # the gather above saved the indices, not the weights, so the in-place update cannot disturb backward
            # (the reference writes embedding.weight.data for the same reason)
            self.ema_step(latent.detach(), indices)
        return x_q, loss, indices.view(x.shape[:-1])

    @torch.no_grad()
    def ema_step(self, latent, indices):
        """The EMA step, the step count and the dead-code reset when it is due (vq.py:146-187, :188-190).  Under
        ``dist_ema`` the step runs over the global batch, and a rank whose block is empty still calls this with 0 rows."""
        if self.dist_ema is None:
            ops.ema_update(latent, indices, self._ema_cluster_size, self._ema_w, self.embedding.weight.data,
                           self.ema_decay, self.epsilon)
            self.step_count += 1
            if self.step_count % self.reset_interval == 0:
                self._reset_unused_codes(latent)
            return
        latent_global = self.dist_ema.update(latent, indices, None, self._ema_cluster_size, self._ema_w,
                                             self.embedding.weight.data, self.ema_decay, self.epsilon)
        self.step_count += 1
        if self.step_count % self.reset_interval == 0:
            self._reset_unused_codes_dist(latent_global)

    @torch.no_grad()
    def _reset_unused_codes_dist(self, latent_global):
        """The reset over the global batch.  The dead codes follow from _ema_cluster_size, identical on every rank, so every
        rank knows whether one happens; rank 0 then draws it (the reference's randint / randperm / randn_like sequence)
        and broadcasts the level's buffers.  Replica equality never rests on the ranks' RNG states agreeing."""
        import torch.distributed as dist
        _, unused_mask = ops.codebook_usage(self._ema_cluster_size, self.epsilon, self.reset_threshold, want_unused=True)
        if int(unused_mask.sum().item()) == 0 or len(latent_global) == 0:
            return
        group = self.dist_ema.group
        if self.dist_ema.rank == 0:
            self._reset_unused_codes(latent_global)
        src = dist.get_global_rank(group, 0) if group is not dist.group.WORLD else 0
        for t in (self.embedding.weight.data, self._ema_cluster_size, self._ema_w):
            dist.broadcast(t, src=src, group=group)

    @torch.no_grad()
    def get_codebook_usage(self):
        used_codes, _ = ops.codebook_usage(self._ema_cluster_size, self.epsilon, self.reset_threshold)
        return {"utilization": used_codes / self.n_e, "used_codes": used_codes, "total_codes": self.n_e}
