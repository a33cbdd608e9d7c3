"""MLP stack, k-means initialiser and Sinkhorn entry point with the reference's import surface.

Mirrors ``index/models/layers.py`` of the reference (``MLPLayers`` :7-43, ``activation_layer``
:45-67, ``kmeans`` :69-82, ``sinkhorn_algorithm`` :85-108): same constructor arguments, same
sub-module layout (so ``state_dict`` keys ``mlp_layers.{i}.weight`` ... are interchangeable with
reference checkpoints), but the arithmetic runs in liblcrec_b200.so:

* inference (no autograd): the whole stack is one ``MlpHandle`` - fp32-accurate split-operand tcgen05 GEMMs with
  fused bias + ReLU, activations handed from layer to layer already split; eval-mode BatchNorm is folded
  into the weights;
* training: each ``nn.Linear`` (+ReLU when nothing sits between them) goes through the same GEMM
  kernel inside an autograd Function; training-mode BatchNorm1d (+ReLU) runs on its own reduce / apply kernels
  (``_BnReluFn``, synchronised over a process group on request); Dropout / non-ReLU activations stay torch modules.

CUDA only - a CPU tensor raises (no fallback).
"""
from __future__ import annotations

import os
from typing import List, Optional

import torch
import torch.nn as nn

from .. import ops


def activation_layer(activation_name="relu", emb_dim=None):
    """Activation factory, same accepted names / errors as reference layers.py:45-67."""
    if activation_name is None:
        return None
    if isinstance(activation_name, str):
        table = {"sigmoid": nn.Sigmoid, "tanh": nn.Tanh, "relu": nn.ReLU, "leakyrelu": nn.LeakyReLU, "none": None}
        key = activation_name.lower()
        ctor = table.get(key)            # unknown strings give None, as in the reference
        return ctor() if ctor is not None else None
    if isinstance(activation_name, type) and issubclass(activation_name, nn.Module):
        return activation_name()
    raise NotImplementedError("activation function {} is not implemented".format(activation_name))


class _LinearFn(torch.autograd.Function):
    """y = relu?(x W^T + b): forward and backward (ReLU mask, bias gradient, gx = g W, gw = g^T x) on the
    fp32-accurate split-operand tcgen05 kernels (lcrec_linear_forward / lcrec_linear_backward)."""

    @staticmethod
    def forward(ctx, x, weight, bias, fuse_relu: bool):
        y = ops.linear_forward(x, weight, bias, fuse_relu)
        ctx.fuse_relu = fuse_relu
        ctx.save_for_backward(x, weight, y if fuse_relu else None)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        x, weight, y = ctx.saved_tensors
        gx, gw, gb = ops.linear_backward(x, weight, y if ctx.fuse_relu else None, gy,
                                         need_gx=ctx.needs_input_grad[0], need_gw=ctx.needs_input_grad[1],
                                         need_gb=ctx.has_bias and ctx.needs_input_grad[2])
        return gx, gw, gb, None


class _BnReluFn(torch.autograd.Function):
    """Training-mode BatchNorm1d + the ReLU behind it (reference layers.py:25-29) on the kernels of csrc/train_extra.cu:
    batch statistics, running-statistics update (momentum / cumulative average exactly like torch), analytic backward.
    ``bn.lcrec_sync = (group, n_total)`` (set by the data-parallel trainer) all-reduces the per-channel sums over the ranks."""

    @staticmethod
    def forward(ctx, y, gamma, beta, bn, relu: bool):
        sync = getattr(bn, "lcrec_sync", None)
        group, n_total = sync if sync is not None else (None, None)
        if (n_total if n_total is not None else y.shape[0]) == 1:   # F.batch_norm's check, on the global batch
            raise ValueError(f"Expected more than 1 value per channel when training, got input size {y.size()}")
        factor = 0.0
        rm = rv = None
        if bn.track_running_stats and bn.running_mean is not None:
            rm, rv = bn.running_mean, bn.running_var
            if bn.num_batches_tracked is not None:
                bn.num_batches_tracked.add_(1)
            if bn.momentum is None:                              # cumulative moving average: needs the count on the host
                factor = 1.0 / float(bn.num_batches_tracked.item())
            else:
                factor = float(bn.momentum)
        out, mean, invstd = ops.bn_relu_forward(y, gamma, beta, rm, rv, factor, bn.eps, relu, group=group, n_total=n_total)
        if rm is not None:                                       # written through raw pointers: version-keyed caches must see it
            from ..optim import _bump_versions
            _bump_versions([rm, rv])
        ctx.save_for_backward(y, out if relu else None, gamma, mean, invstd)
        ctx.relu, ctx.sync = relu, (group, n_total)
        return out

    @staticmethod
    def backward(ctx, gy):
        y, out, gamma, mean, invstd = ctx.saved_tensors
        need_gp = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        gx, gg, gb = ops.bn_relu_backward(y, gy, out, ctx.relu, gamma, mean, invstd, need_gx=ctx.needs_input_grad[0],
                                          need_gp=need_gp, group=ctx.sync[0], n_total=ctx.sync[1])
        return gx, (gg if ctx.needs_input_grad[1] else None), (gb if ctx.needs_input_grad[2] else None), None, None


class _MlpFn(torch.autograd.Function):
    """A whole Linear/ReLU stack as ONE autograd node: forward = lcrec_mlp_forward (activations kept for the backward),
    backward = lcrec_mlp_backward (one native loop over the layers).  Used in training when nothing but ReLU sits
    between the Linear layers (no BatchNorm, no active Dropout)."""

    @staticmethod
    def forward(ctx, x, handle, n_layers, *params):
        y, acts = handle.forward(x, want_acts=True)
        ctx.handle = handle
        ctx.save_for_backward(x, *acts)
        ctx.has_bias = [params[2 * i + 1] is not None for i in range(n_layers)]
        return y

    @staticmethod
    def backward(ctx, gy):
        x, *acts = ctx.saved_tensors
        gx, gws, gbs = ctx.handle.backward(x, acts, gy, need_gx=ctx.needs_input_grad[0])
        grads = []
        for i, (gw, gb) in enumerate(zip(gws, gbs)):
            grads.append(gw if ctx.needs_input_grad[3 + 2 * i] else None)
            grads.append(gb if (ctx.has_bias[i] and ctx.needs_input_grad[4 + 2 * i]) else None)
        return (gx, None, None, *grads)


class MLPLayers(nn.Module):
    def __init__(self, layers, dropout=0.0, activation="relu", bn=False):
        super().__init__()
        self.layers = layers
        self.dropout = dropout
        self.activation = activation
        self.use_bn = bn

        mods: List[nn.Module] = []
        n_lin = len(layers) - 1
        for i in range(n_lin):
            mods.append(nn.Dropout(p=dropout))
            mods.append(nn.Linear(layers[i], layers[i + 1]))
            if i != n_lin - 1:
                if bn:
                    mods.append(nn.BatchNorm1d(num_features=layers[i + 1]))
                act = activation_layer(activation, layers[i + 1])
                if act is not None:
                    mods.append(act)
        self.mlp_layers = nn.Sequential(*mods)
        self.apply(self.init_weights)
        self._handle: Optional[ops.MlpHandle] = None
        self._handle_key = None

    def init_weights(self, module):
        if isinstance(module, nn.Linear):           # Xavier-normal W, zero b (reference layers.py:35-40)
            nn.init.xavier_normal_(module.weight.data)
            if module.bias is not None:
                module.bias.data.fill_(0.0)

    # ------------------------------------------------------------------ structure helpers
    def _blocks(self):
        """[(dropout, linear, bn|None, act|None)] in order."""
        blocks, cur = [], None
        for m in self.mlp_layers:
            if isinstance(m, nn.Dropout):
                if cur is not None:
                    blocks.append(cur)
                cur = [m, None, None, None]
            elif isinstance(m, nn.Linear):
                cur[1] = m
            elif isinstance(m, nn.BatchNorm1d):
                cur[2] = m
            else:
                cur[3] = m
        blocks.append(cur)
        return blocks

    def _fused_ok(self, input_feature=None) -> bool:
        """The no-autograd handle path serves the call only when nothing needs a gradient: neither a parameter nor the
        INPUT (a frozen stack in front of a trainable one must still propagate d/dx like nn.Sequential would)."""
        if torch.is_grad_enabled() and (any(p.requires_grad for p in self.parameters())
                                        or (input_feature is not None and input_feature.requires_grad)):
            return False
        blocks = self._blocks()
        for i, (dp, lin, bn, act) in enumerate(blocks):
            last = i == len(blocks) - 1
            if self.training and (dp.p > 0 or bn is not None):
                return False
            if not last and not isinstance(act, nn.ReLU):
                return False
            if lin.out_features % 4 != 0 and last:
                return False
        return True

    def _folded(self):
        """(weights, biases) with eval-mode BatchNorm folded in (computed in fp64, rounded once)."""
        ws, bs = [], []
        for dp, lin, bn, act in self._blocks():
            w = lin.weight.detach()
            b = lin.bias.detach() if lin.bias is not None else torch.zeros(lin.out_features, device=w.device)
            if bn is not None:
                inv = 1.0 / torch.sqrt(bn.running_var.double() + bn.eps)
                g = bn.weight.detach().double() if bn.affine else torch.ones_like(inv)
                beta = bn.bias.detach().double() if bn.affine else torch.zeros_like(inv)
                s = g * inv
                w = (w.double() * s[:, None]).float()
                b = ((b.double() - bn.running_mean.double()) * s + beta).float()
            ws.append(w)
            bs.append(b)
        return ws, bs

    def _get_handle(self) -> ops.MlpHandle:
        key = tuple((t.data_ptr(), t._version) for t in list(self.parameters()) + list(self.buffers()))
        if self._handle is None or self._handle_key != key:
            ws, bs = self._folded()
            if self._handle is not None and self._handle.device == ws[0].device:
                self._handle.update(ws, bs)
            else:
                self._handle = ops.MlpHandle(ws, bs, relu_last=False)
            self._handle_key = key
        return self._handle

    def _stack_ok(self) -> bool:
        """Training with autograd, and the stack is Linear(+ReLU) only: one fused autograd node serves it."""
        blocks = self._blocks()
        for i, (dp, lin, bn, act) in enumerate(blocks):
            last = i == len(blocks) - 1
            if bn is not None or (self.training and dp.p > 0) or lin.bias is None:
                return False
            if (not last and not isinstance(act, nn.ReLU)) or (last and act is not None):
                return False
            if lin.out_features % 4 != 0 or lin.in_features % 4 != 0:
                return False
        return True

    def forward(self, input_feature):
        if not input_feature.is_cuda:
            raise RuntimeError("lcrec_b200.MLPLayers runs on CUDA only (no CPU fallback)")
        if self._fused_ok(input_feature):
            return self._get_handle().forward(input_feature)
        if self._stack_ok():
            handle = self._get_handle()
            params = []
            for dp, lin, bn, act in self._blocks():
                params += [lin.weight, lin.bias]
            lead = input_feature.shape[:-1]
            y = _MlpFn.apply(input_feature.reshape(-1, input_feature.shape[-1]), handle, len(params) // 2, *params)
            return y.reshape(*lead, y.shape[-1])
        x = input_feature
        blocks = self._blocks()
        for i, (dp, lin, bn, act) in enumerate(blocks):
            x = dp(x)
            fuse = bn is None and isinstance(act, nn.ReLU)
            x = _LinearFn.apply(x, lin.weight, lin.bias, fuse)
            if bn is not None:
                if bn.training or not bn.track_running_stats:     # batch statistics: the BN + ReLU kernels
                    fuse = isinstance(act, nn.ReLU)
                    lead = x.shape
                    x = _BnReluFn.apply(x.reshape(-1, lead[-1]), bn.weight, bn.bias, bn, fuse).reshape(lead)
                else:
                    x = bn(x)                                     # eval statistics with autograd on (not a training path)
            if act is not None and not fuse:
                x = act(x)
        return x


# "sklearn": the reference's own call, bit-reproducible against it.  "device": k-means++ seeding by scikit-learn on the host
# (same draws from numpy's global RNG as KMeans.fit), Lloyd iterations in liblcrec_b200.so (lcrec_kmeans_lloyd).
KMEANS_BACKEND = os.environ.get("LCREC_KMEANS", "sklearn")


def kmeans(samples, num_clusters, num_iters=10):
    """Codebook initialisation (reference layers.py:69-82: sklearn ``KMeans(n_clusters, max_iter).fit`` on the CPU copy).

    Backend "sklearn" delegates exactly as the reference does.  Backend "device" keeps only the k-means++ seeding on the
    host - ``sklearn.cluster.kmeans_plusplus`` on the centred batch consumes numpy's global RNG exactly like ``fit`` (tested)
    - and runs sklearn's Lloyd loop (centring, tol = 1e-4 x mean column variance, strict / tol stop, empty-cluster
    relocation, final E-step) on the device; centres agree with sklearn's to fp32 rounding whenever the label sequences
    coincide (tests/test_gpu_zz_kmeans.py)."""
    if KMEANS_BACKEND == "sklearn":
        from sklearn.cluster import KMeans
        x = samples.detach().cpu().numpy()
        fit = KMeans(n_clusters=num_clusters, max_iter=num_iters).fit(x)
        return torch.from_numpy(fit.cluster_centers_).to(samples.device)
    if KMEANS_BACKEND not in ("device", "device_seed"):
        raise ValueError(f"unknown k-means backend {KMEANS_BACKEND!r}")
    xc, mean, mean_var = ops.kmeans_center(samples.detach())
    if KMEANS_BACKEND == "device":
        from sklearn.cluster import kmeans_plusplus
        seeds, _ = kmeans_plusplus(xc.cpu().numpy(), num_clusters)
        seeds = torch.from_numpy(seeds).to(xc.device)
    else:
        # "device_seed" (not yet run on hardware in round 1): the seeding on the device as well; the host only DRAWS the
        # random numbers, in sklearn's order, from numpy's global RNG (their count does not depend on the data)
        first, draws = kmeanspp_random_numbers(xc.shape[0], num_clusters)
        _, seeds = ops.kmeanspp_seed(xc, num_clusters, first, torch.from_numpy(draws))
    fit = ops.kmeans_lloyd(xc, seeds, num_iters, 1e-4 * mean_var, add_mean=mean)
    return fit["centers"]


def kmeanspp_random_numbers(n_samples, num_clusters):
    """What ``sklearn.cluster.kmeans_plusplus`` draws from numpy's global RNG, in its order: the first centre through
    ``RandomState.choice(n, p=uniform)`` (one uniform -> searchsorted on the normalised cumulative weights, side 'right'),
    then ``uniform(size=2 + int(log(K)))`` per further centre.  Returns (first index, (K-1, trials) fp64)."""
    import numpy as np
    rs = np.random.mtrand._rand
    trials = 2 + int(np.log(num_clusters))
    w = np.ones(n_samples, dtype=np.float32)                      # sklearn's unit sample weights, in the data's dtype
    p = (w / w.sum()).astype(np.float64)                          # RandomState.choice converts p to double
    cdf = p.cumsum()
    cdf /= cdf[-1]
    first = int(cdf.searchsorted(rs.random_sample(), side="right"))
    draws = np.stack([rs.uniform(size=trials) for _ in range(1, num_clusters)]) if num_clusters > 1 else np.zeros((0, trials))
    return first, draws


@torch.no_grad()
def sinkhorn_algorithm(distances, epsilon, sinkhorn_iterations):
    """Drop-in for reference layers.py:85-108 on a CUDA tensor: returns the transport plan Q with
    the reference's literal normalisation order, computed by the fp64 cooperative kernel.  Inputs
    that are not fp64 are promoted (fp32 overflows at eps=0.003) and the result cast back."""
    q = ops.sinkhorn_dense(distances, float(epsilon), int(sinkhorn_iterations))
    return q if distances.dtype == torch.float64 else q.to(distances.dtype)
