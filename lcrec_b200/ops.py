"""Tensor-level wrappers over the C ABI.  torch provides device memory and streams only; every
computation below happens inside liblcrec_b200.so (hand-written sm_100a kernels)."""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib


def _stream(t: torch.Tensor) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _need_cuda(*ts: torch.Tensor) -> None:
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("lcrec_b200 operators run on a CUDA (sm_100a) device only; there is no CPU "
                               f"fallback (got a tensor on {t.device})")


def _f32c(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(torch.float32).contiguous()


def _p(t: Optional[torch.Tensor]) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


def _ws(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


import os as _os

# GEMM operand encoding used by every MlpHandle created afterwards: 1 = f16 x3 (default), 0 = tf32 x3.
DEFAULT_ENGINE = int(_os.environ.get("LCREC_ENGINE", "1"))


def set_default_engine(engine: int) -> None:
    global DEFAULT_ENGINE
    assert engine in (0, 1)
    DEFAULT_ENGINE = int(engine)


def launch_count() -> int:
    return int(_lib.load().lcrec_launch_count())


def sinkhorn_set_mode(mode: int) -> None:
    """0 = literal in-place divides everywhere; 1 = scaling-vector form; 2 = filtered hybrid (default):
    scaling form + literal re-run of every group whose argmax is not provably the literal one."""
    _lib.check(_lib.load().lcrec_sinkhorn_set_mode(int(mode)))


def fp64_peak_tflops(device=None) -> float:
    """Measured DFMA peak of the device in TFLOP/s (lcrec_fp64_peak_probe)."""
    dev = torch.device(device or f"cuda:{torch.cuda.current_device()}")
    ws = torch.empty(8 * 2048 * 256, dtype=torch.uint8, device=dev)
    out = C.c_double()
    with torch.cuda.device(dev):
        _lib.check(_lib.load().lcrec_fp64_peak_probe(C.byref(out), _p(ws), ws.numel(), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return out.value / 1e12


def sinkhorn_set_col(on) -> None:
    """A/B switch of the column kernels (lcrec_sinkhorn_set_col): False / 0 = off, 1 = groups of 9..32 rows only, True / 2 (default)
    = also every group of a call with few groups (late collision rounds); results are identical."""
    _lib.check(_lib.load().lcrec_sinkhorn_set_col(2 if on is True else int(on)))


def ddiv_probe(a: torch.Tensor, b: torch.Tensor):
    """(wrong, fallback) of lcrec_ddiv_probe over the fp64 device pairs (a[i], b[i]): quotients of the shared-reciprocal
    division that differ from the device's IEEE a / b (must be 0) and pairs its range check hands to the fallback."""
    assert a.is_cuda and a.dtype == torch.float64 and b.dtype == torch.float64 and a.numel() == b.numel()
    a, b = a.contiguous(), b.contiguous()
    counts = torch.zeros(2, dtype=torch.int64, device=a.device)
    with torch.cuda.device(a.device):
        _lib.check(_lib.load().lcrec_ddiv_probe(_p(a), _p(b), a.numel(), _p(counts), C.c_void_p(torch.cuda.current_stream(a.device).cuda_stream)))
    w, f = counts.tolist()
    return int(w), int(f)


def profile_enable(on: bool) -> None:
    _lib.check(_lib.load().lcrec_profile_enable(int(on)))


def profile_collect() -> dict:
    """{tag: (ms, calls)} accumulated since the last collect (synchronises the device)."""
    ms = (C.c_double * 32)()
    calls = (C.c_int64 * 32)()
    _lib.check(_lib.load().lcrec_profile_collect(ms, calls))
    return {t: (ms[t], int(calls[t])) for t in range(32) if calls[t]}


# --------------------------------------------------------------------------- host-visible status words
# The reference reads two device flags on the host inside VectorQuantizer.forward (the Python `assert` of vq.py:59 and the
# NaN/Inf print of vq.py:81-82).  By default they are read where the reference reads them.  A training loop can wrap its
# step in `defer_checks()`: the flags are queued and evaluated by `flush_checks()` at the end of the step (where the
# reference loop synchronises anyway for `loss.item()`), so the forward pass enqueues without draining the GPU.
_DEFER = False
_PENDING: List[Tuple[str, torch.Tensor]] = []


def _evaluate_check(kind: str, word: torch.Tensor) -> None:
    v = int(word.item())
    if kind == "amplitude" and v != 0:
        raise AssertionError("amplitude > 0")
    if kind == "sinkhorn":
        if v & 8:
            raise RuntimeError("distributed Sinkhorn: a peer rank did not arrive")
        if v & 1:
            print("Sinkhorn Algorithm returns nan/inf values.")


def check_later(kind: str, word: torch.Tensor) -> None:
    if _DEFER:
        _PENDING.append((kind, word))
    else:
        _evaluate_check(kind, word)


def take_pending() -> List[Tuple[str, torch.Tensor]]:
    """Hand the queued status words to the caller WITHOUT reading them (a step captured in a CUDA graph keeps the tensors
    and evaluates them after each replay)."""
    pending, _PENDING[:] = list(_PENDING), []
    return pending


def evaluate_check_value(kind: str, v: int) -> None:
    """The check of `_evaluate_check` on a value that is already on the host."""
    if kind == "amplitude" and v != 0:
        raise AssertionError("amplitude > 0")
    if kind == "sinkhorn":
        if v & 8:
            raise RuntimeError("distributed Sinkhorn: a peer rank did not arrive")
        if v & 1:
            print("Sinkhorn Algorithm returns nan/inf values.")


def flush_checks() -> None:
    pending, _PENDING[:] = list(_PENDING), []
    for kind, word in pending:
        _evaluate_check(kind, word)


class defer_checks:
    def __enter__(self):
        global _DEFER
        self._old, _DEFER = _DEFER, True
        return self

    def __exit__(self, *exc):
        global _DEFER
        _DEFER = self._old
        if exc[0] is None and not _DEFER:
            flush_checks()
        elif exc[0] is not None:
            _PENDING.clear()
        return False


# --------------------------------------------------------------------------- MLP
class MlpHandle:
    """Prepared (hi/lo-split) weights of one MLPLayers stack."""

    def __init__(self, weights: Sequence[torch.Tensor], biases: Sequence[Optional[torch.Tensor]],
                 relu_last: bool = False):
        _need_cuda(*weights)
        self.lib = _lib.load()
        self.device = weights[0].device
        self.dims = [int(weights[0].shape[1])] + [int(w.shape[0]) for w in weights]
        self.n_layers = len(weights)
        self.handle = C.c_void_p()
        ws, bs = self._pack(weights, biases)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.lcrec_mlp_create(self.n_layers, _lib.i32_array(self.dims), ws, bs, int(relu_last),
                                                 _stream(weights[0]), C.byref(self.handle)))
        self._workspace: Optional[torch.Tensor] = None
        self.set_engine(DEFAULT_ENGINE)

    def _pack(self, weights, biases):
        self._keep = [_f32c(w) for w in weights]
        self._keepb = [None if b is None else _f32c(b) for b in biases]
        for w, (fi, fo) in zip(self._keep, zip(self.dims[:-1], self.dims[1:])):
            assert tuple(w.shape) == (fo, fi)
        return (_lib.ptr_array([w.data_ptr() for w in self._keep]),
                _lib.ptr_array([0 if b is None else b.data_ptr() for b in self._keepb]))

    def update(self, weights, biases) -> None:
        ws, bs = self._pack(weights, biases)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.lcrec_mlp_update(self.handle, ws, bs, _stream(self._keep[0])))

    def set_acc_chunk(self, k_elems: int) -> None:
        _lib.check(self.lib.lcrec_mlp_set_acc_chunk(self.handle, int(k_elems)))

    def set_engine(self, engine: int) -> None:
        """0 = tf32 x3, 1 = f16 x3 (see include/lcrec_b200.h)."""
        _lib.check(self.lib.lcrec_mlp_set_engine(self.handle, int(engine)))

    def set_variant(self, v: int) -> None:
        _lib.check(self.lib.lcrec_mlp_set_variant(self.handle, int(v)))

    def set_trace(self, buf: Optional[torch.Tensor]) -> None:
        """Measurement only: int64 CUDA tensor of 4*512*4 elements receiving pipeline clock stamps, or None."""
        self._trace = buf
        _lib.check(self.lib.lcrec_mlp_set_trace(self.handle, _p(buf)))

    def forward(self, x: torch.Tensor, want_acts: bool = False):
        _need_cuda(x)
        x2 = _f32c(x.reshape(-1, self.dims[0]))
        n = x2.shape[0]
        y = torch.empty((n, self.dims[-1]), dtype=torch.float32, device=x2.device)
        need = int(self.lib.lcrec_mlp_workspace_bytes(self.handle, n))
        if self._workspace is None or self._workspace.numel() < need or self._workspace.device != x2.device:
            if self._workspace is not None:                  # a captured CUDA graph may still point at the old one
                self.__dict__.setdefault("_retired", []).append(self._workspace)
            self._workspace = _ws(need, x2.device)
        acts = None
        acts_arr = None
        if want_acts:
            acts = [torch.empty((n, d), dtype=torch.float32, device=x2.device) for d in self.dims[1:-1]] + [y]
            acts_arr = _lib.ptr_array([a.data_ptr() for a in acts])
        with torch.cuda.device(x2.device):
            _lib.check(self.lib.lcrec_mlp_forward(self.handle, _p(x2), n, _p(y), acts_arr, _p(self._workspace),
                                                  self._workspace.numel(), _stream(x2)))
        y = y.reshape(*x.shape[:-1], self.dims[-1])
        return (y, acts) if want_acts else y

    def backward(self, x: torch.Tensor, acts: Sequence[torch.Tensor], gy: torch.Tensor, need_gx: bool = True):
        """Gradients of the whole stack (lcrec_mlp_backward): returns (gx or None, [gw_l], [gb_l]).  ``acts`` as returned
        by ``forward(x, want_acts=True)``; the weights are the ones of the last ``update`` / construction."""
        _need_cuda(x, gy)
        x2 = _f32c(x.reshape(-1, self.dims[0]))
        g2 = _f32c(gy.reshape(-1, self.dims[-1]))
        n = x2.shape[0]
        dev = x2.device
        gx = torch.empty((n, self.dims[0]), dtype=torch.float32, device=dev) if need_gx else None
        gws = [torch.empty((fo, fi), dtype=torch.float32, device=dev) for fi, fo in zip(self.dims[:-1], self.dims[1:])]
        gbs = [torch.empty((fo,), dtype=torch.float32, device=dev) for fo in self.dims[1:]]
        ws = _ws(self.lib.lcrec_mlp_backward_workspace_bytes(self.handle, n), dev)
        with torch.cuda.device(dev):
            _lib.check(self.lib.lcrec_mlp_backward(self.handle, _lib.ptr_array([w.data_ptr() for w in self._keep]), _p(x2),
                                                   _lib.ptr_array([a.data_ptr() for a in acts]), _p(g2), n, _p(gx),
                                                   _lib.ptr_array([g.data_ptr() for g in gws]),
                                                   _lib.ptr_array([g.data_ptr() for g in gbs]), _p(ws), ws.numel(), _stream(x2)))
        return (None if gx is None else gx.reshape(x.shape)), gws, gbs

    def __del__(self):
        try:
            if self.handle:
                self.lib.lcrec_mlp_destroy(self.handle)
                self.handle = C.c_void_p()
        except Exception:
            pass


def linear_forward(x: torch.Tensor, w: torch.Tensor, b: Optional[torch.Tensor], relu: bool,
                   acc_chunk: int = 64, variant: Optional[int] = None) -> torch.Tensor:
    """relu?(x @ w.T + b) with the split-operand tcgen05 kernel (nn.Linear, layers.py:23).
    variant: bit 0 = alternative tile, bit 1 = f16 x3 engine, bits 1+2 (6) = CTA-pair kernel; default: the module-wide
    DEFAULT_ENGINE, on the pair kernel where the shape allows."""
    if variant is None:
        variant = 2 * DEFAULT_ENGINE
        m_, k_ = int(w.shape[0]), int(w.shape[1])
        if DEFAULT_ENGINE == 1 and (m_ % 256 == 0 or m_ in (128, 64)) and k_ >= 64 and k_ % 8 == 0:
            variant = 6                      # CTA-pair kernel (same rule as linear_pair_supported in csrc/linear_pair.cu)
    _need_cuda(x, w)
    lib = _lib.load()
    x2, w2 = _f32c(x.reshape(-1, w.shape[1])), _f32c(w)
    b2 = None if b is None else _f32c(b)
    n, k, m = x2.shape[0], w2.shape[1], w2.shape[0]
    y = torch.empty((n, m), dtype=torch.float32, device=x2.device)
    ws = _ws(lib.lcrec_linear_workspace_bytes(n, k, m), x2.device)
    with torch.cuda.device(x2.device):
        _lib.check(lib.lcrec_linear_forward(_p(x2), n, k, _p(w2), _p(b2), m, int(relu), _p(y), int(acc_chunk),
                                            int(variant), _p(ws), ws.numel(), _stream(x2)))
    return y.reshape(*x.shape[:-1], m)


def linear_backward(x: torch.Tensor, w: torch.Tensor, y_relu: Optional[torch.Tensor], gy: torch.Tensor,
                    need_gx: bool = True, need_gw: bool = True, need_gb: bool = True):
    """Gradients of relu?(x @ w.T + b) (autograd of nn.Linear + ReLU, trainer.py:114-118) on the split-operand
    tensor-core kernels: returns (gx, gw, gb), None for the ones not requested."""
    _need_cuda(x, w, gy)
    lib = _lib.load()
    m, k = w.shape
    x2, w2, g2 = _f32c(x.reshape(-1, k)), _f32c(w), _f32c(gy.reshape(-1, m))
    y2 = None if y_relu is None else _f32c(y_relu.reshape(-1, m))
    n = x2.shape[0]
    gx = torch.empty((n, k), dtype=torch.float32, device=x2.device) if need_gx else None
    gw = torch.empty((m, k), dtype=torch.float32, device=x2.device) if need_gw else None
    gb = torch.empty((m,), dtype=torch.float32, device=x2.device) if need_gb else None
    ws = _ws(lib.lcrec_linear_backward_workspace_bytes(n, k, m), x2.device)
    with torch.cuda.device(x2.device):
        _lib.check(lib.lcrec_linear_backward(_p(x2), _p(w2), _p(y2), _p(g2), n, k, m, _p(gx), _p(gw), _p(gb), _p(ws),
                                             ws.numel(), _stream(x2)))
    return (None if gx is None else gx.reshape(x.shape)), gw, gb


# --------------------------------------------------------------------------- BatchNorm (training) + reconstruction loss
def bn_relu_forward(y: torch.Tensor, gamma: Optional[torch.Tensor], beta: Optional[torch.Tensor],
                    running_mean: Optional[torch.Tensor], running_var: Optional[torch.Tensor], momentum: float, eps: float,
                    relu: bool, group=None, n_total: Optional[int] = None):
    """Training-mode ``BatchNorm1d`` (+ the ReLU behind it, layers.py:25-29) of a (n, C) Linear output: returns
    (out, save_mean, save_invstd) and updates the running statistics in place.  ``group``: all-reduce the per-channel sums
    over a process group (synchronised BN; ``n_total`` = the global row count, known to the caller)."""
    _need_cuda(y)
    lib = _lib.load()
    y2 = _f32c(y)
    n, c = y2.shape
    sums = torch.empty(int(lib.lcrec_bn_sums_elems(c)), dtype=torch.float64, device=y2.device)
    out = torch.empty_like(y2)
    mean = torch.empty(c, dtype=torch.float32, device=y2.device)
    invstd = torch.empty(c, dtype=torch.float32, device=y2.device)
    splits = int(lib.lcrec_bn_splits(n, c))
    with torch.cuda.device(y2.device):
        _lib.check(lib.lcrec_bn_forward_reduce(_p(y2), n, c, _p(sums), _stream(y2)))
        if group is not None:
            import torch.distributed as dist
            red = sums[: splits * 2 * c].view(splits, 2 * c).sum(0)
            dist.all_reduce(red, group=group)
            sums[: 2 * c] = red
            splits = 1
        tot = int(n_total) if n_total is not None else n
        _lib.check(lib.lcrec_bn_forward_apply(_p(y2), _p(sums), splits, n, tot, c, _p(gamma), _p(beta), float(eps), float(momentum),
                                              int(relu), _p(out), _p(mean), _p(invstd), _p(running_mean), _p(running_var), _stream(y2)))
    return out, mean, invstd


def bn_relu_backward(y: torch.Tensor, gy: torch.Tensor, out: torch.Tensor, relu: bool, gamma: Optional[torch.Tensor],
                     mean: torch.Tensor, invstd: torch.Tensor, need_gx: bool = True, need_gp: bool = True, group=None,
                     n_total: Optional[int] = None):
    """(gx, g_gamma, g_beta) of the training-mode BatchNorm1d + ReLU above."""
    _need_cuda(y, gy)
    lib = _lib.load()
    y2, g2 = _f32c(y), _f32c(gy)
    n, c = y2.shape
    sums = torch.empty(int(lib.lcrec_bn_sums_elems(c)), dtype=torch.float64, device=y2.device)
    gx = torch.empty_like(y2) if need_gx else None
    gg = torch.empty(c, dtype=torch.float32, device=y2.device) if need_gp else None
    gb = torch.empty(c, dtype=torch.float32, device=y2.device) if need_gp else None
    splits = int(lib.lcrec_bn_splits(n, c))
    with torch.cuda.device(y2.device):
        _lib.check(lib.lcrec_bn_backward_reduce(_p(y2), _p(g2), _p(out), int(relu), _p(mean), _p(invstd), n, c, _p(sums), _stream(y2)))
        if group is not None:
            # synchronised BN: gx needs the sums over the GLOBAL batch; g_gamma / g_beta stay this rank's LOCAL sums, because the
            # trainer's gradient all-reduce (SUM over ranks) adds them up afterwards like every other parameter gradient
            import torch.distributed as dist
            red = sums[: splits * 2 * c].view(splits, 2 * c).sum(0)
            if need_gp:
                gb, gg = red[:c].to(torch.float32), red[c:].to(torch.float32)
            dist.all_reduce(red, group=group)
            sums[: 2 * c] = red
            splits = 1
        tot = int(n_total) if n_total is not None else n
        _lib.check(lib.lcrec_bn_backward_apply(_p(y2), _p(g2), _p(out), int(relu), _p(sums), splits, n, tot, c, _p(gamma), _p(mean),
                                               _p(invstd), _p(gx), _p(None if group is not None else gg),
                                               _p(None if group is not None else gb), _stream(y2)))
    return gx, gg, gb


_LOSS_TYPES = {"mse": 0, "l1": 1}


def recon_loss(out: torch.Tensor, x: torch.Tensor, loss_type: str) -> torch.Tensor:
    """``F.mse_loss`` / ``F.l1_loss`` (reduction="mean") of rqvae.py:74-85 as a 0-dim fp32 tensor."""
    _need_cuda(out, x)
    lib = _lib.load()
    o2, x2 = _f32c(out), _f32c(x)
    assert o2.shape == x2.shape
    loss = torch.empty((), dtype=torch.float32, device=o2.device)
    ws = _ws(lib.lcrec_recon_loss_workspace_bytes(o2.numel()), o2.device)
    with torch.cuda.device(o2.device):
        _lib.check(lib.lcrec_recon_loss(_p(o2), _p(x2), o2.numel(), _LOSS_TYPES[loss_type], _p(loss), _p(ws), ws.numel(), _stream(o2)))
    return loss


def recon_loss_backward(out: torch.Tensor, x: torch.Tensor, loss_type: str, upstream: Optional[torch.Tensor]) -> torch.Tensor:
    _need_cuda(out, x)
    lib = _lib.load()
    o2, x2 = _f32c(out), _f32c(x)
    grad = torch.empty_like(o2)
    up = None if upstream is None else upstream.detach().to(torch.float32).contiguous()
    with torch.cuda.device(o2.device):
        _lib.check(lib.lcrec_recon_loss_backward(_p(o2), _p(x2), o2.numel(), _LOSS_TYPES[loss_type], _p(up), _p(grad), _stream(o2)))
    return grad.view(out.shape)


# --------------------------------------------------------------------------- RQ
def rq_set_tc_mode(mode: int) -> None:
    """0 = SIMT kernels only, 1 = tensor-core distance GEMM for large codebooks (default), 2 = whenever possible."""
    _lib.check(_lib.load().lcrec_rq_set_tc_mode(int(mode)))


def rq_quantize(z: torch.Tensor, codebooks: Sequence[torch.Tensor], n_levels_run: Optional[int] = None,
                resid_level: int = -1, want_codes: bool = True, want_xq: bool = False,
                want_sq_err: bool = False):
    """Fused argmin residual quantisation over ``codebooks[:n_levels_run]`` (rq.py:39-56).

    Returns dict with codes (n, L_run) int64, xq (n, D), resid (residual entering ``resid_level``;
    ``resid_level == n_levels_run`` gives the residual left after the last level run), sq_err (L_run) fp64.
    """
    _need_cuda(z, *codebooks)
    lib = _lib.load()
    d = int(codebooks[0].shape[1])
    z2 = _f32c(z.reshape(-1, d))
    n = z2.shape[0]
    cbs = [_f32c(c) for c in codebooks]
    run = len(cbs) if n_levels_run is None else int(n_levels_run)
    cbs = cbs[:max(run, 1)]
    L = len(cbs)
    dev = z2.device
    codes = torch.empty((n, L), dtype=torch.int64, device=dev) if want_codes else None
    xq = torch.empty((n, d), dtype=torch.float32, device=dev) if want_xq else None
    resid = torch.empty((n, d), dtype=torch.float32, device=dev) if resid_level >= 0 else None
    err = torch.zeros((L,), dtype=torch.float64, device=dev) if want_sq_err else None
    with torch.cuda.device(dev):
        _lib.check(lib.lcrec_rq_quantize(_p(z2), n, d, L, _lib.ptr_array([c.data_ptr() for c in cbs]),
                                         _lib.i32_array([c.shape[0] for c in cbs]), run, int(resid_level), _p(codes),
                                         _p(xq), _p(resid), _p(err), _stream(z2)))
    if codes is not None and run < L:
        codes = codes[:, :run]
    return {"codes": codes, "xq": xq, "resid": resid, "sq_err": err}


def rq_train_forward(z: torch.Tensor, codes: torch.Tensor, codebooks: Sequence[torch.Tensor]):
    """Forward values of the residual quantiser for given codes (rq.py:39-56): dict(xq (n, D), diffs (L, n, D),
    codes_t (L, n), sq_err (L) fp64)."""
    _need_cuda(z, codes, *codebooks)
    lib = _lib.load()
    cbs = [_f32c(c) for c in codebooks]
    L, d = len(cbs), int(cbs[0].shape[1])
    z2 = _f32c(z.reshape(-1, d))
    n = z2.shape[0]
    c2 = codes.detach().reshape(n, L).to(torch.int64).contiguous()
    dev = z2.device
    xq = torch.empty((n, d), dtype=torch.float32, device=dev)
    diffs = torch.empty((L, n, d), dtype=torch.float32, device=dev)
    codes_t = torch.empty((L, n), dtype=torch.int64, device=dev)
    err = torch.empty((L,), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.lcrec_rq_train_forward(_p(z2), _p(c2), n, d, L, _lib.ptr_array([c.data_ptr() for c in cbs]), _p(xq),
                                              _p(diffs), _p(codes_t), _p(err), _stream(z2)))
    return {"xq": xq, "diffs": diffs, "codes_t": codes_t, "sq_err": err}


def rq_train_backward(diffs: torch.Tensor, codes_t: torch.Tensor, n_codes: Sequence[int], g_xq: Optional[torch.Tensor],
                      g_loss: Optional[torch.Tensor], beta0: float, want_gz: bool = True, want_gcb: bool = True):
    """Analytic backward of (x_q, mean level loss) w.r.t. (z, codebooks); see include/lcrec_b200.h."""
    _need_cuda(diffs, codes_t, g_xq, g_loss)
    lib = _lib.load()
    L, n, d = diffs.shape
    dev = diffs.device
    gx = None if g_xq is None else _f32c(g_xq.reshape(n, d))
    gl = None if g_loss is None else _f32c(g_loss.reshape(1))
    gz = torch.empty((n, d), dtype=torch.float32, device=dev) if want_gz else None
    gcbs = [torch.empty((int(k), d), dtype=torch.float32, device=dev) for k in n_codes] if want_gcb else None
    with torch.cuda.device(dev):
        _lib.check(lib.lcrec_rq_train_backward(
            _p(diffs), _p(codes_t), n, d, L, _lib.i32_array(list(n_codes)), _p(gx), _p(gl), float(beta0), _p(gz),
            _lib.ptr_array([g.data_ptr() for g in gcbs]) if want_gcb else None, _stream(diffs)))
    return gz, gcbs


def vq_distances(r: torch.Tensor, codebook: torch.Tensor) -> torch.Tensor:
    """(n, K) fp32 distances of vq.py:71-73."""
    _need_cuda(r, codebook)
    lib = _lib.load()
    cb = _f32c(codebook)
    r2 = _f32c(r.reshape(-1, cb.shape[1]))
    out = torch.empty((r2.shape[0], cb.shape[0]), dtype=torch.float32, device=r2.device)
    with torch.cuda.device(r2.device):
        _lib.check(lib.lcrec_vq_distances(_p(r2), r2.shape[0], cb.shape[1], _p(cb), cb.shape[0], _p(out), _stream(r2)))
    return out


# --------------------------------------------------------------------------- k-means initialisation
def kmeans_center(x: torch.Tensor):
    """(x - column means, means, mean of the column variances): the frame sklearn's KMeans.fit works in."""
    _need_cuda(x)
    lib = _lib.load()
    x2 = _f32c(x.reshape(-1, x.shape[-1]))
    n, d = x2.shape
    xc = torch.empty_like(x2)
    mean = torch.empty(d, dtype=torch.float32, device=x2.device)
    var = C.c_double(0.0)
    ws = _ws(lib.lcrec_kmeans_workspace_bytes(n, d, 1), x2.device)
    with torch.cuda.device(x2.device):
        _lib.check(lib.lcrec_kmeans_center(_p(x2), n, d, _p(xc), _p(mean), C.byref(var), _p(ws), ws.numel(), _stream(x2)))
    return xc, mean, float(var.value)


def kmeanspp_seed(xc: torch.Tensor, n_clusters: int, first_index: int, draws: torch.Tensor):
    """k-means++ seeds of sklearn's `_kmeans_plusplus` on centred rows from pre-drawn uniforms (``draws``: (K-1, trials)
    fp64).  Returns (indices (K,) int64, centers (K, D))."""
    _need_cuda(xc)
    lib = _lib.load()
    x2 = _f32c(xc)
    n, d = x2.shape
    dr = draws.detach().to(device=x2.device, dtype=torch.float64).contiguous()
    if dr.numel():
        dr = dr.reshape(n_clusters - 1, -1)
    trials = int(dr.shape[1]) if dr.numel() else 1
    idx = torch.empty(n_clusters, dtype=torch.int64, device=x2.device)
    centers = torch.empty((n_clusters, d), dtype=torch.float32, device=x2.device)
    ws = _ws(lib.lcrec_kmeanspp_workspace_bytes(n, trials), x2.device)
    with torch.cuda.device(x2.device):
        _lib.check(lib.lcrec_kmeanspp_seed(_p(x2), n, d, int(n_clusters), int(first_index), _p(dr) if dr.numel() else None,
                                           trials, _p(idx), _p(centers), _p(ws), ws.numel(), _stream(x2)))
    return idx, centers


def kmeans_lloyd(xc: torch.Tensor, seeds: torch.Tensor, max_iter: int, tol: float, add_mean: Optional[torch.Tensor] = None):
    """Lloyd iterations from ``seeds`` on centred data -> dict(centers, labels, inertia, n_iter) (sklearn semantics)."""
    _need_cuda(xc, seeds, add_mean)
    lib = _lib.load()
    x2 = _f32c(xc)
    n, d = x2.shape
    centers = _f32c(seeds).clone()
    k = centers.shape[0]
    labels = torch.empty(n, dtype=torch.int64, device=x2.device)
    inertia, n_iter = C.c_double(0.0), C.c_int(0)
    ws = _ws(lib.lcrec_kmeans_workspace_bytes(n, d, k), x2.device)
    am = None if add_mean is None else _f32c(add_mean)
    with torch.cuda.device(x2.device):
        _lib.check(lib.lcrec_kmeans_lloyd(_p(x2), n, d, _p(centers), k, int(max_iter), float(tol), _p(am), _p(labels),
                                          C.byref(inertia), C.byref(n_iter), _p(ws), ws.numel(), _stream(x2)))
    return {"centers": centers, "labels": labels, "inertia": float(inertia.value), "n_iter": int(n_iter.value)}


# --------------------------------------------------------------------------- EMA codebook variant
def _inplace_f32(t: torch.Tensor, name: str) -> torch.Tensor:
    if t.dtype != torch.float32 or not t.is_contiguous():
        raise RuntimeError(f"{name} must be a contiguous fp32 tensor (it is updated in place)")
    return t


def ema_update(latent: torch.Tensor, indices: torch.Tensor, cluster_size: torch.Tensor, ema_w: torch.Tensor,
               codebook: torch.Tensor, ema_decay: float, epsilon: float) -> None:
    """EMA step of index_improve/models/vq.py:146-187, in place on (cluster_size, ema_w, codebook)."""
    _need_cuda(latent, indices, cluster_size, ema_w, codebook)
    lib = _lib.load()
    k, d = codebook.shape
    lat = _f32c(latent.reshape(-1, d))
    idx = indices.detach().reshape(-1).to(torch.int64).contiguous()
    if idx.shape[0] != lat.shape[0]:
        raise RuntimeError("ema_update: one index per latent row expected")
    _inplace_f32(cluster_size, "cluster_size"); _inplace_f32(ema_w, "ema_w"); _inplace_f32(codebook, "codebook")
    with torch.cuda.device(lat.device):
        _lib.check(lib.lcrec_ema_update(_p(lat), _p(idx), lat.shape[0], k, d, float(ema_decay), float(epsilon),
                                        _p(cluster_size), _p(ema_w), _p(codebook), _stream(lat)))


def codebook_usage(cluster_size: torch.Tensor, epsilon: float, reset_threshold: float, want_unused: bool = False):
    """(used_codes, unused_mask or None) of index_improve/models/vq.py:205-217 / :83-87."""
    _need_cuda(cluster_size)
    lib = _lib.load()
    cs = _f32c(cluster_size)
    used = torch.zeros(1, dtype=torch.int64, device=cs.device)
    mask = torch.empty(cs.shape[0], dtype=torch.uint8, device=cs.device) if want_unused else None
    with torch.cuda.device(cs.device):
        _lib.check(lib.lcrec_codebook_usage(_p(cs), cs.shape[0], float(epsilon), float(reset_threshold), _p(used),
                                            _p(mask), _stream(cs)))
    return int(used.item()), (mask.bool() if want_unused else None)


# --------------------------------------------------------------------------- embedding producer hand-off
# element type codes of the C ABI's `dtype` arguments: the hidden states of the pool, the embeddings of the _ex indexer entries
DTYPE_CODES = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}


def masked_mean_pool(last_hidden_state: torch.Tensor, attention_mask: torch.Tensor, out: Optional[torch.Tensor] = None,
                     accumulate: bool = False, divide_by: float = 0.0) -> torch.Tensor:
    """``(h * mask[..., None]).sum(1) / mask.sum(-1, keepdim=True)`` (data_process/amazon_text_emb.py:91-92) -> fp32
    (B, H).  ``out``: fp32 rows to write (a view into the embedding matrix; row stride >= H, unit column stride);
    ``accumulate`` adds to ``out``; ``divide_by`` > 0 divides the result (mean over text fields, :96)."""
    _need_cuda(last_hidden_state, attention_mask, out)
    lib = _lib.load()
    if last_hidden_state.dtype not in DTYPE_CODES:
        raise RuntimeError(f"masked_mean_pool: unsupported hidden dtype {last_hidden_state.dtype}")
    h = last_hidden_state.detach().contiguous()
    b, t, d = h.shape
    m = attention_mask.detach().to(torch.int64).contiguous()
    if m.shape != (b, t):
        raise RuntimeError("masked_mean_pool: attention_mask must be (batch, seq_len)")
    if out is None:
        if accumulate:
            raise RuntimeError("masked_mean_pool: accumulate needs an existing out")
        out = torch.empty((b, d), dtype=torch.float32, device=h.device)
    if out.dtype != torch.float32 or out.shape != (b, d) or (d > 1 and out.stride(1) != 1) or out.device != h.device:
        raise RuntimeError("masked_mean_pool: out must be fp32 (batch, hidden) with unit column stride on the same device")
    stride = out.stride(0) if b > 1 else max(d, out.stride(0))
    ws = _ws(lib.lcrec_masked_mean_pool_workspace_bytes(b, t, d), h.device)
    with torch.cuda.device(h.device):
        _lib.check(lib.lcrec_masked_mean_pool(_p(h), DTYPE_CODES[h.dtype], _p(m), b, t, d, _p(out), stride,
                                              int(accumulate), float(divide_by), _p(ws), ws.numel(), _stream(h)))
    return out


# --------------------------------------------------------------------------- Sinkhorn
def center_distances(d: torch.Tensor) -> torch.Tensor:
    """center_distance_for_constraint (vq.py:51-61) followed by .double() (vq.py:78)."""
    _need_cuda(d)
    lib = _lib.load()
    d2 = _f32c(d)
    out = torch.empty(d2.shape, dtype=torch.float64, device=d2.device)
    status = torch.zeros(1, dtype=torch.int32, device=d2.device)
    ws = _ws(16384, d2.device)
    with torch.cuda.device(d2.device):
        _lib.check(lib.lcrec_center_distances(_p(d2), d2.shape[0], d2.shape[1], _p(out), _p(status), _p(ws),
                                              ws.numel(), _stream(d2)))
    check_later("amplitude", status)                # vq.py:59 (a host read; deferred to the end of the step under defer_checks)
    return out


def sinkhorn_dense(distances: torch.Tensor, epsilon: float, iters: int, want_argmax: bool = False):
    """sinkhorn_algorithm (layers.py:85-108) on a CUDA fp64 matrix; optional fused argmax (vq.py:83)."""
    _need_cuda(distances)
    lib = _lib.load()
    d = distances.detach().to(torch.float64).contiguous()
    b, k = d.shape
    q = torch.empty_like(d)
    arg = torch.empty((b,), dtype=torch.int64, device=d.device) if want_argmax else None
    flags = torch.zeros(1, dtype=torch.int32, device=d.device)
    ws = _ws(lib.lcrec_sinkhorn_workspace_bytes(b, k), d.device)
    with torch.cuda.device(d.device):
        _lib.check(lib.lcrec_sinkhorn_dense(_p(d), b, k, float(epsilon), int(iters), _p(q), _p(arg), _p(flags), _p(ws),
                                            ws.numel(), _stream(d)))
    return (q, arg, flags) if want_argmax else q


def sinkhorn_dense_argmax(distances: torch.Tensor, epsilon: float, iters: int):
    """``argmax(sinkhorn_algorithm(distances, epsilon, iters), -1)`` (vq.py:78-83) without materialising the plan: one
    thread-block cluster with the kernel matrix in distributed shared memory (lcrec_sinkhorn_dense_argmax).
    Returns (indices int64 (B,), flags int32 (1,))."""
    _need_cuda(distances)
    lib = _lib.load()
    d = distances.detach().to(torch.float64).contiguous()
    b, k = d.shape
    arg = torch.empty((b,), dtype=torch.int64, device=d.device)
    flags = torch.zeros(1, dtype=torch.int32, device=d.device)
    ws = _ws(lib.lcrec_sinkhorn_dense_argmax_workspace_bytes(b, k), d.device)
    with torch.cuda.device(d.device):
        _lib.check(lib.lcrec_sinkhorn_dense_argmax(_p(d), b, k, float(epsilon), int(iters), _p(arg), _p(flags), _p(ws), ws.numel(),
                                                   _stream(d)))
    return arg, flags


def sinkhorn_set_wide(on) -> None:
    """Large-codebook path of the per-group Sinkhorn (batched distances + one cluster per group); False / 0 = CTA kernel only,
    2 = the cluster path with the literal divide form for every group (cross-check of the re-run kernel)."""
    _lib.check(_lib.load().lcrec_sinkhorn_set_wide(int(on)))


def sinkhorn_set_dense_cluster(on: bool) -> None:
    _lib.check(_lib.load().lcrec_sinkhorn_set_dense_cluster(int(bool(on))))


def collisions(codes: torch.Tensor, n_codes: Sequence[int]):
    """Sort/unique over packed code tuples -> CSR collision groups + counts (generate_indices.py:18-42)."""
    _need_cuda(codes)
    lib = _lib.load()
    c = codes.detach().to(torch.int64).contiguous()
    n, L = c.shape
    dev = c.device
    offsets = torch.empty((n + 1,), dtype=torch.int64, device=dev)
    members = torch.empty((max(n, 1),), dtype=torch.int64, device=dev)
    counts = torch.zeros((4,), dtype=torch.int64, device=dev)
    ws = _ws(lib.lcrec_collisions_workspace_bytes(n), dev)
    with torch.cuda.device(dev):
        _lib.check(lib.lcrec_collisions(_p(c), n, L, _lib.i32_array(n_codes), _p(offsets), _p(members), _p(counts),
                                        _p(ws), ws.numel(), _stream(c)))
    n_unique, n_groups, n_rows, max_mult = [int(v) for v in counts.tolist()]
    return {"offsets": offsets[: n_groups + 1], "members": members[:n_rows], "n_unique": n_unique,
            "n_groups": n_groups, "n_rows": n_rows, "max_multiplicity": max_mult, "counts_dev": counts}


def prefix_segments(codes: torch.Tensor, n_codes: Sequence[int]):
    """Runs (>= 2 items) of equal first L-1 codes, CSR like ``collisions`` (members ordered by (last code, item))."""
    _need_cuda(codes)
    lib = _lib.load()
    c = codes.detach().to(torch.int64).contiguous()
    n, L = c.shape
    dev = c.device
    offsets = torch.empty((n + 1,), dtype=torch.int64, device=dev)
    members = torch.empty((max(n, 1),), dtype=torch.int64, device=dev)
    counts = torch.zeros((8,), dtype=torch.int64, device=dev)
    ws = _ws(lib.lcrec_collisions_workspace_bytes(n), dev)
    with torch.cuda.device(dev):
        _lib.check(lib.lcrec_prefix_segments(_p(c), n, L, _lib.i32_array(n_codes), _p(offsets), _p(members), _p(counts),
                                             _p(ws), ws.numel(), _stream(c)))
    _, n_segs, n_rows, max_size = [int(v) for v in counts[:4].tolist()]
    return {"offsets": offsets[: n_segs + 1], "members": members[:n_rows], "n_segments": n_segs, "n_rows": n_rows,
            "max_size": max_size, "counts_dev": counts}


def collisions_in_segments(codes: torch.Tensor, segs: dict, level: Optional[int] = None):
    """Collision groups of the current codes searched inside prefix segments (no global sort); same result dict as
    ``collisions`` plus ``fallback`` (True: a segment exceeded the on-chip sort, use ``collisions``)."""
    _need_cuda(codes)
    lib = _lib.load()
    c = codes.detach().to(torch.int64).contiguous()
    n, L = c.shape
    dev = c.device
    level = L - 1 if level is None else level
    offsets = torch.empty((n + 1,), dtype=torch.int64, device=dev)
    members = torch.empty((max(n, 1),), dtype=torch.int64, device=dev)
    counts = torch.zeros((8,), dtype=torch.int64, device=dev)
    max_segs = segs["n_segments"]
    ws = _ws(lib.lcrec_segment_collisions_workspace_bytes(max_segs), dev)
    with torch.cuda.device(dev):
        _lib.check(lib.lcrec_collisions_in_segments(_p(c), n, L, int(level), _p(segs["offsets"]), _p(segs["members"]),
                                                    _p(segs["counts_dev"][1:2]), max_segs, _p(offsets), _p(members),
                                                    _p(counts), _p(ws), ws.numel(), _stream(c)))
    vals = [int(v) for v in counts.tolist()]
    n_unique, n_groups, n_rows, max_mult = vals[:4]
    return {"offsets": offsets[: n_groups + 1], "members": members[:n_rows], "n_unique": n_unique, "n_groups": n_groups,
            "n_rows": n_rows, "max_multiplicity": max_mult, "counts_dev": counts, "fallback": bool(vals[5])}


def indexer_set_segments(on: bool) -> None:
    _lib.check(_lib.load().lcrec_indexer_set_segments(int(bool(on))))


def indexer_set_speculative(mode) -> None:
    """Later collision rounds: 0 / False = one host read per round, 1 = all remaining rounds enqueued blind on the caller's stream,
    2 / True (default) = late rounds (<= 888 groups) replayed from a CUDA graph in batches; identical results."""
    _lib.check(_lib.load().lcrec_indexer_set_speculative(2 if mode is True else int(mode)))


def sort_codes(codes: torch.Tensor, n_codes: Sequence[int]):
    _need_cuda(codes)
    lib = _lib.load()
    c = codes.detach().to(torch.int64).contiguous()
    n, L = c.shape
    keys = torch.empty((n,), dtype=torch.int64, device=c.device)
    items = torch.empty((n,), dtype=torch.int32, device=c.device)
    ws = _ws(lib.lcrec_collisions_workspace_bytes(n), c.device)
    with torch.cuda.device(c.device):
        _lib.check(lib.lcrec_sort_codes(_p(c), n, L, _lib.i32_array(n_codes), _p(keys), _p(items), _p(ws), ws.numel(),
                                        _stream(c)))
    return keys, items


def sinkhorn_groups(resid: torch.Tensor, codebook: torch.Tensor, offsets: torch.Tensor, members: torch.Tensor,
                    n_groups_dev: torch.Tensor, max_groups: int, max_rows: int, epsilon: float, iters: int,
                    codes: torch.Tensor, level: int, part_mod: int = 1, part_rem: int = 0, want_risky: bool = False):
    """Per-group Sinkhorn re-assignment of ``codes[:, level]`` in place; returns the flag word (and, on
    request, how many groups the filtered mode re-ran through the literal kernel)."""
    _need_cuda(resid, codebook, offsets, members, codes)
    lib = _lib.load()
    assert codes.dtype == torch.int64 and codes.is_contiguous()
    r, cb = _f32c(resid), _f32c(codebook)
    flags = torch.zeros(2, dtype=torch.int32, device=r.device)
    ws = _ws(lib.lcrec_sinkhorn_groups_workspace_bytes(max_rows, cb.shape[0]), r.device)
    with torch.cuda.device(r.device):
        _lib.check(lib.lcrec_sinkhorn_groups_part(_p(r), cb.shape[1], _p(cb), cb.shape[0], _p(offsets), _p(members),
                                                  _p(n_groups_dev), int(max_groups), int(max_rows), float(epsilon),
                                                  int(iters), _p(codes), codes.shape[1], int(level), int(part_mod),
                                                  int(part_rem), _p(flags), _p(ws), ws.numel(), _stream(r)))
    if want_risky:   # the library keeps its cursor words at the start of the workspace: [big cursor u64][risky count i32]
        off = (-ws.data_ptr()) % 256
        return int(flags[0].item()), int(ws[off + 8: off + 12].view(torch.int32).item())
    return int(flags[0].item())


def index_json_bytes(codes: torch.Tensor) -> bytes:
    """The `.index.json` text of a CUDA code table (n, L) int64 - the bytes ``json.dump`` writes at
    generate_indices.py:144-145 - formatted on the device (lcrec_index_json) and copied to the host once."""
    _need_cuda(codes)
    lib = _lib.load()
    c = codes.detach().to(torch.int64).contiguous()
    n, L = c.shape
    total = torch.zeros(1, dtype=torch.int64, device=c.device)
    ws = _ws(lib.lcrec_index_json_workspace_bytes(n), c.device)
    cap = 2 + n * (2 + 1 + 20 + 1 + 2 + 2 + L * (6 + 20 + 2))          # generous upper bound; most of it is never touched
    if n <= 4_000_000:
        cap = 2 + n * (2 + 1 + 7 + 1 + 2 + 2 + L * (6 + 20 + 2))
    out = torch.empty(cap, dtype=torch.uint8, device=c.device)
    with torch.cuda.device(c.device):
        _lib.check(lib.lcrec_index_json(_p(c), n, L, _p(out), cap, _p(total), _p(ws), ws.numel(), _stream(c)))
    nbytes = int(total.item())
    assert nbytes <= cap
    return out[:nbytes].cpu().numpy().tobytes()


# --------------------------------------------------------------------------- whole generation
_HALF = (torch.float16, torch.bfloat16)


def _embeddings(x: torch.Tensor) -> Tuple[torch.Tensor, Optional[int]]:
    """(tensor, dtype code) for the indexer entries: fp16 / bf16 embeddings stay as they are (contiguous; the kernels read
    them natively, code 1 / 2); every other dtype becomes an fp32 copy as before (code None: the fp32 entry)."""
    if x.dtype in _HALF:
        return x.detach().contiguous(), DTYPE_CODES[x.dtype]
    return _f32c(x), None


class Indexer:
    """generate_indices.py:85-128 on the device (PASS 0 + collision rounds)."""

    def __init__(self, encoder: MlpHandle, codebooks: Sequence[torch.Tensor], last_epsilon: float, sk_iters: int,
                 max_items: int, chunk_rows: int = 131072):
        self.lib = _lib.load()
        self.encoder = encoder
        self.cbs = [_f32c(c) for c in codebooks]
        _need_cuda(*self.cbs)
        self.L = len(self.cbs)
        self.D = int(self.cbs[0].shape[1])
        self.device = self.cbs[0].device
        self.max_items = int(max_items)
        self.handle = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.lcrec_indexer_create(encoder.handle, self.D, self.L,
                                                     _lib.ptr_array([c.data_ptr() for c in self.cbs]),
                                                     _lib.i32_array([c.shape[0] for c in self.cbs]), float(last_epsilon),
                                                     int(sk_iters), self.max_items, int(chunk_rows), C.byref(self.handle)))

    def _stats(self, raw) -> dict:
        keys = ["rounds", "n_unique", "groups_round1", "rows_round1", "sinkhorn_rows", "max_multiplicity", "nan_flag"]
        return {k: int(raw[i]) for i, k in enumerate(keys)}

    def run_device(self, x: torch.Tensor, max_rounds: int = 20) -> Tuple[torch.Tensor, dict]:
        """x: CUDA (n, in_dim) embeddings.  fp16 / bf16 are read as they are (no fp32 copy); the codes and stats are
        those of the fp32 run on ``x.float()``, bit for bit."""
        _need_cuda(x)
        x2, code = _embeddings(x)
        n = x2.shape[0]
        codes = torch.empty((n, self.L), dtype=torch.int64, device=x2.device)
        stats = (C.c_int64 * 8)()
        with torch.cuda.device(x2.device):
            if code is None:
                _lib.check(self.lib.lcrec_indexer_run_device(self.handle, _p(x2), n, int(max_rounds), _p(codes), stats,
                                                             _stream(x2)))
            else:
                _lib.check(self.lib.lcrec_indexer_run_device_ex(self.handle, _p(x2), code, n, int(max_rounds), _p(codes),
                                                                stats, _stream(x2)))
        return codes, self._stats(stats)

    def run_host(self, x_host, codes_host=None, max_rounds: int = 20):
        """x_host: CPU float32 / float16 / bfloat16 tensor or ndarray (n, in_dim), contiguous (pinned or pageable); half
        precision is copied to the device as it is (half the bytes).  Returns CPU int64 codes."""
        xt = torch.as_tensor(x_host)
        assert not xt.is_cuda and xt.dtype in (torch.float32,) + _HALF and xt.is_contiguous()
        n = xt.shape[0]
        out = torch.empty((n, self.L), dtype=torch.int64) if codes_host is None else codes_host
        stats = (C.c_int64 * 8)()
        with torch.cuda.device(self.device):
            st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
            if xt.dtype == torch.float32:
                _lib.check(self.lib.lcrec_indexer_run_host(self.handle, C.c_void_p(xt.data_ptr()), n, int(max_rounds),
                                                           C.c_void_p(out.data_ptr()), stats, st))
            else:
                _lib.check(self.lib.lcrec_indexer_run_host_ex(self.handle, C.c_void_p(xt.data_ptr()), DTYPE_CODES[xt.dtype], n,
                                                              int(max_rounds), C.c_void_p(out.data_ptr()), stats, st))
        return out, self._stats(stats)

    def resolve_device(self, codes: torch.Tensor, resid: torch.Tensor, max_rounds: int = 20) -> dict:
        """The collision rounds alone on caller-owned tensors (codes updated in place)."""
        _need_cuda(codes, resid)
        assert codes.dtype == torch.int64 and codes.is_contiguous() and resid.dtype == torch.float32 and resid.is_contiguous()
        stats = (C.c_int64 * 8)()
        with torch.cuda.device(codes.device):
            _lib.check(self.lib.lcrec_indexer_resolve(self.handle, _p(codes), _p(resid), codes.shape[0], int(max_rounds),
                                                      stats, _stream(codes)))
        return self._stats(stats)

    def pass0(self, x: torch.Tensor, row_offset: int = 0) -> None:
        x2, code = _embeddings(x)
        with torch.cuda.device(x2.device):
            if code is None:
                _lib.check(self.lib.lcrec_indexer_pass0(self.handle, _p(x2), x2.shape[0], int(row_offset), _stream(x2)))
            else:
                _lib.check(self.lib.lcrec_indexer_pass0_ex(self.handle, _p(x2), code, x2.shape[0], int(row_offset),
                                                           _stream(x2)))

    def round(self, n: int) -> dict:
        counts = (C.c_int64 * 4)()
        with torch.cuda.device(self.device):
            st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
            _lib.check(self.lib.lcrec_indexer_round(self.handle, int(n), counts, st))
        return {"n_unique": int(counts[0]), "n_groups": int(counts[1]), "n_rows": int(counts[2]),
                "max_multiplicity": int(counts[3])}

    def _view(self, ptr: int, shape, dtype) -> torch.Tensor:
        import numpy as np  # local: only for the dtype size
        n = 1
        for s in shape:
            n *= s
        itemsize = torch.empty((), dtype=dtype).element_size()
        # wrap borrowed device memory without copying (torch has no public from-pointer; use __cuda_array_interface__)
        class _Holder:
            pass
        h = _Holder()
        typestr = {torch.int64: "<i8", torch.float32: "<f4"}[dtype]
        h.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 3}
        return torch.as_tensor(h, device=self.device)

    def codes_view(self, n: int) -> torch.Tensor:
        return self._view(self.lib.lcrec_indexer_codes(self.handle), (n, self.L), torch.int64)

    def resid_view(self, n: int) -> torch.Tensor:
        return self._view(self.lib.lcrec_indexer_resid(self.handle), (n, self.D), torch.float32)

    def __del__(self):
        try:
            if self.handle:
                self.lib.lcrec_indexer_destroy(self.handle)
                self.handle = C.c_void_p()
        except Exception:
            pass
