"""Training-step kernels of csrc/train_extra.cu and csrc/optim.cu element by element against fp64 (B200).

u = 2^-24, E = 2^-53, TINY = 2^-149 (one fp32 subnormal step).  Every bound below is a first-order rounding analysis of
the kernel's own operation sequence; the C constants are set at about 4x the worst ratio measured on a B200 (DESIGN.md
sections 2.2 and 4.8).  Each case prints its worst |err| / bound; a failure names the first element over its bound.

BatchNorm1d(train) [+ ReLU] forward (`bn_reduce_kernel<false>` + `bn_apply_kernel`).  Reference on the fp32 input y in
fp64, two-pass: m = mean(y), v = mean((y - m)^2), is = 1 / sqrt(v + eps), x = (y - m) is, out64 = relu?(g x + b)
(eps the fp32 value the kernel adds).  The kernel sums y and y^2 in fp64 in chains of at most
L = ceil(ceil(n / S) / 8) + 8 + S adds (S row splits of 8 lanes, then the 8 lanes, then the splits), takes
var = sum(y^2) / n - m^2 (one pass), rounds m and is once to fp32 and evaluates (y - mu) is g + b in fp32.  With
VAR = (L + 1) E (m^2 + v) / (v + eps), the worst case of the one-pass variance is a relative error 4 VAR in v, 2 VAR in is:

    |out - out64| <= C_BN u (|g| is (|y - m| + |m|) + |g x| + |b|)  +  K_VAR VAR |g x|  +  (|g| is + 1) TINY
    |save_mean - m| <= ulp32(m) + L E mean|y|          |save_invstd - is| <= (C_BN u + K_VAR VAR) is + TINY

(the |g| is |m| term is the fp32 rounding of the saved mean, which torch shares).  The worst case of C_BN is about 4 and
of K_VAR 2.  VAR stays below u up to |m| / sigma = 2^20 at every tested n: that is the supported range, asserted on
offset channels 2^0 .. 2^20; offsets 2^21 .. 2^24 are asserted finite and their ratio is printed.  Channels of
magnitude 2^-120 .. 2^120, constant channels, a 2^20 sigma outlier row, mixed-sign and zero gamma share the bound.
Running statistics after two steps (momentum 0.1 and None = cumulative average) against torch's rule in fp64 with the
unbiased factor n / (n - 1): per step, err' = (1 - f) err + C_RUN (u ((1 - f)|r| + f|s| + |r'|) + f ERR_s) with
ERR_s = u |m| for the mean and (u + 4 VAR) |s| for the variance.

Backward, teacher-forced on the kernel's out (ReLU mask), save_mean and save_invstd: x = (y - mean) invstd in fp64,
gm = g [out > 0], g_beta = sum gm, g_gamma = sum gm x, gx64 = gamma invstd (gm - g_beta / N - x g_gamma / N):

    |gx - gx64| <= C_BWD u |gamma invstd| (|gm| + |g_beta| / N + |x| sum |gm x| / N) + TINY
    |g_beta - g_beta64| <= C_BWD u sum |gm| + TINY,     |g_gamma - g_gamma64| <= C_BWD u sum |gm x| + TINY

The kernel rounds its x to fp32 per element (2u), so the g_gamma it divides by N is off by up to 2u sum |gm x|, which
can be far more than 2u |g_gamma| where sum gm x cancels: |x g_gamma| / N in place of |x| sum |gm x| / N fails on
random row-spread gradients (measured 9.3 x 8u on a B200).

Synchronised BatchNorm runs the real `group` branch of ops.bn_relu_forward / bn_relu_backward on one GPU with
torch.distributed.all_reduce replaced by a record / replay pair over R ragged virtual ranks; the concatenated result is
held to the same bounds for the global batch (L grows by S + R for the extra additions).

Exact (bit for bit): column permutation, y -> 2^e y at eps = 0 (out, g_gamma, g_beta unchanged; save_mean x 2^e,
save_invstd and gx x 2^-e), constant channel -> relu(beta), gamma / beta None == ones / zeros, repeat calls, and a NaN
or +-inf at (r, c) poisons channel c only, forward and backward.

Reconstruction loss: |loss - L64| <= C_LOSS u L64 + TINY with L64 the fp64 mean of (o - x)^2 or |o - x| (all terms >= 0;
worst case about 6 u); the gradient equals the fp32 replay fl(fl(fl(2 fl(1/N)) up) fl(o - x)) (mse) or
fl(fl(1 fl(1/N)) up) sign(o - x) with sign(NaN) = 0 (l1) bit for bit, also for inputs that are not 16-byte aligned.

Optimisers (47 tensors, sizes around the 4096-element CTA chunk, gradient scales 2^-40 .. 2^40): total norm within
C_NORM u of the fp64 sqrt(sum g^2); the written-back gradient equals fl(g coef), coef = min(1, fl(max_norm /
fl(norm + 1e-6f))) replayed from the returned norm, bit for bit; without clipping the gradients are untouched.  Adam /
AdamW / SGD / Adagrad / RMSprop state and parameters are teacher-forced on the clipped gradient and evaluated in fp64 with
the fp32 hyper-parameters the kernel uses (lcrec_adam_hyper); the bound is C_OPT times the propagated first-order error
of the kernel's line sequence, each fp32 rounding of a result r contributing u |r| + TINY and a square root
min(e / (2 sqrt(s)), sqrt(e)) of an input error e (the worst case of C_OPT is 1)."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from lcrec_b200 import _lib, ops
    from lcrec_b200.models.layers import MLPLayers, _BnReluFn
    from lcrec_b200.optim import FusedAdam, FusedSimple
    DEV = torch.device("cuda:0")

U = 2.0 ** -24
E53 = 2.0 ** -53
TINY = 2.0 ** -149
# Bound constants (module docstring), about 4x the worst ratio measured on a B200 (DESIGN.md sections 2.2, 4.8).
C_BN = 7.0             # measured 1.66 (out of 4097 x 2048, relu; the offset channels' mean rounding)
K_VAR = 2.0            # the worst case of the one-pass variance (not separable from C_BN in a measurement)
C_RUN = 8.0            # measured 2.03 (synchronised running_mean, R = 2)
C_BWD = 16.0           # measured 4.0 (gx, 4097 x 2048, relu, row-spread gradients; g_gamma 1.84)
C_LOSS = 2.25          # measured 0.55 (mse, 2^24 + 3 elements 2^+-60)
C_NORM = 3.5           # measured 0.85 (47 tensors, scales 2^+-40)
C_OPT = 4.0            # measured 0.9998: one rounding reaching its half ulp (adamw m, step 2)
EPS = float(np.float32(1e-5))          # BatchNorm1d's eps as the kernel adds it (fp32)
SUPPORTED = 20                         # |m| / sigma up to 2^SUPPORTED is held to the bound


def report(capsys, name, ratio, what="|err| / bound"):
    with capsys.disabled():
        print(f"\n  [{name}] worst {what} = {ratio:.3e}")


def check_elements(capsys, name, y, y64, bnd, show=True):
    """|y - y64| <= bnd everywhere (prints the worst ratio first, then names the first offender); returns the ratio"""
    err = (y.double() - y64).abs()
    ratio = float(torch.where(err == 0, torch.zeros_like(err), err / bnd).max()) if err.numel() else 0.0
    if show or not ratio <= 1:
        report(capsys, name, ratio)
    bad = ~(err <= bnd)
    if bad.any():
        i = tuple(bad.nonzero()[0].tolist())
        raise AssertionError(f"{name}: {int(bad.sum())} elements over the bound, first {list(i)}: got={y[i].item()!r} "
                             f"ref={y64[i].item()!r} bound={bnd[i].item()!r}")
    return ratio


def bits(t):
    return t.contiguous().view(torch.int32)


def same_bits(a, b):
    """bit-identical, NaN == NaN whatever the payload"""
    if a.shape != b.shape:
        return False
    nan = torch.isnan(a)
    return bool(torch.equal(nan, torch.isnan(b)) and torch.equal(bits(a)[~nan], bits(b)[~nan]))


def gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def f32(x):
    return float(np.float32(x))


# ================================================================== BatchNorm
def bn_splits(n, c):
    """bn_splits() of csrc/train_extra.cu: 16 at most, 2 CTAs per SM over the channel blocks, >= 64 rows per split"""
    sms = torch.cuda.get_device_properties(DEV).multi_processor_count
    s = max(1, min(16, (2 * sms) // ((c + 31) // 32)))
    return min(s, max(1, n // 64))


def chain(n, splits):
    return -(-(-(-n // splits)) // 8) + 8 + splits


N_OFFSETS = 25                         # offsets 2^0 .. 2^24
MAGS = list(range(-120, 121, 20))      # magnitude channels 2^-120 .. 2^120 at m = 0
N_KINDS = N_OFFSETS + len(MAGS) + 2    # + constant + outlier


def bn_inputs(n, c, seed):
    """(y, gamma, beta, offset exponent per channel or -1): channel j has kind j mod N_KINDS - an offset channel
    +-2^k sigma (sigma a power of two in 2^-10 .. 2^10), a magnitude channel randn 2^e, a constant channel, or randn with one
    row 2^20 out.  Every 7th gamma is 0, the others mixed-sign."""
    g = gen(seed)
    y = torch.randn(n, c, device=DEV, generator=g, dtype=torch.float64)
    kind = torch.arange(c, device=DEV) % N_KINDS
    sig = torch.exp2(torch.randint(-10, 11, (c,), device=DEV, generator=g).double())
    sgn = torch.where(torch.rand(c, device=DEV, generator=g) < 0.5, -1.0, 1.0).double()
    off = torch.where(kind < N_OFFSETS, kind, torch.full_like(kind, -1))
    mag = torch.tensor(MAGS, device=DEV, dtype=torch.float64)
    is_mag = (kind >= N_OFFSETS) & (kind < N_OFFSETS + len(MAGS))
    scale = torch.where(is_mag, torch.exp2(mag[(kind - N_OFFSETS).clamp(0, len(MAGS) - 1)]), sig)
    shift = torch.where(off >= 0, sgn * torch.exp2(off.double()) * sig, torch.zeros_like(sig))
    y = y * scale + shift
    const = kind == N_OFFSETS + len(MAGS)
    y[:, const] = (torch.randn(int(const.sum()), device=DEV, generator=g, dtype=torch.float64) * 3.0)[None, :]
    outl = kind == N_KINDS - 1
    if n > 1:
        y[n // 2, outl] += 2.0 ** 20 * sig[outl]
    gamma = torch.randn(c, device=DEV, generator=g)
    gamma[::7] = 0
    beta = torch.randn(c, device=DEV, generator=g)
    return y.float(), gamma, beta, off


def bn_fwd_ref(y, gamma, beta, relu, eps=EPS):
    y64 = y.double()
    m = y64.mean(0)
    v = ((y64 - m) ** 2).mean(0)
    inv = 1.0 / torch.sqrt(v + eps)
    ga = torch.ones_like(m) if gamma is None else gamma.double()
    be = torch.zeros_like(m) if beta is None else beta.double()
    x = (y64 - m) * inv
    out = ga * x + be
    return (out.clamp_min(0) if relu else out), m, v, inv, ga, be, x


def var_rel(m, v, L, eps=EPS):
    return (L + 1) * E53 * (m * m + v) / (v + eps)


def check_bn_forward(capsys, name, y, gamma, beta, relu, out, mean, invstd, L, off=None):
    out64, m, v, inv, ga, be, x = bn_fwd_ref(y, gamma, beta, relu)
    vr = var_rel(m, v, L)
    bnd = C_BN * U * (ga.abs() * inv * ((y.double() - m).abs() + m.abs()) + (ga * x).abs() + be.abs()) \
        + K_VAR * vr * (ga * x).abs() + (ga.abs() * inv + 1) * TINY
    sup = torch.ones_like(m, dtype=torch.bool) if off is None else off <= SUPPORTED
    assert torch.isfinite(out).all(), f"{name}: non-finite output"
    check_elements(capsys, name + " out", out[:, sup], out64[:, sup], bnd[:, sup])
    if not bool(sup.all()):
        err = (out.double() - out64).abs()[:, ~sup] / bnd[:, ~sup]
        report(capsys, name + " out, offsets beyond 2^20 (not asserted)", float(err.max()))
    m32 = m.float().abs()
    ulp = (torch.nextafter(m32, torch.full_like(m32, math.inf)) - m32).double()
    check_elements(capsys, name + " save_mean", mean, m, ulp + L * E53 * y.double().abs().mean(0))
    check_elements(capsys, name + " save_invstd", invstd[sup], inv[sup], ((C_BN * U + K_VAR * vr) * inv + TINY)[sup])


# n, C, the split count bn_splits() picks on a 148-SM B200
BN_SHAPES = [(2, 31, 1), (3, 33, 1), (63, 100, 1), (64, 1, 1), (65, 32, 1), (1023, 33, 15), (1024, 32, 16),
             (4097, 100, 16), (4097, 2048, 4), (1024, 4096, 2), (131073, 33, 16)]


@pytest.mark.parametrize("n,c,splits", BN_SHAPES)
@pytest.mark.parametrize("relu", [True, False])
def test_bn_forward_fp64(capsys, n, c, splits, relu):
    lib = _lib.load()
    assert int(lib.lcrec_bn_splits(n, c)) == bn_splits(n, c)
    if torch.cuda.get_device_properties(DEV).multi_processor_count == 148:
        assert bn_splits(n, c) == splits
    y, gamma, beta, off = bn_inputs(n, c, seed=n * 7919 + c)
    out, mean, invstd = ops.bn_relu_forward(y, gamma, beta, None, None, 0.1, EPS, relu)
    check_bn_forward(capsys, f"bn fwd {n}x{c} S={bn_splits(n, c)} relu={relu}", y, gamma, beta, relu, out, mean, invstd,
                     chain(n, bn_splits(n, c)), off)


@pytest.mark.parametrize("momentum", [0.1, None])
@pytest.mark.parametrize("n,c", [(2, 33), (1024, 100), (4097, 2048)])
def test_bn_running_stats_fp64(capsys, momentum, n, c):
    """two training steps through _BnReluFn: torch's update rule with the unbiased factor n / (n - 1); momentum None is the
    cumulative average 1 / num_batches_tracked"""
    bn = torch.nn.BatchNorm1d(c, momentum=momentum).to(DEV).train()
    g = gen(n + c)
    bn.running_mean.copy_(torch.randn(c, device=DEV, generator=g))
    bn.running_var.copy_(torch.rand(c, device=DEV, generator=g) + 0.5)
    rm, rv = bn.running_mean.double().clone(), bn.running_var.double().clone()
    bm = torch.zeros_like(rm)
    bv = torch.zeros_like(rv)
    L = chain(n, bn_splits(n, c))
    for step in range(1, 3):
        y = torch.randn(n, c, device=DEV, generator=g) * (torch.rand(c, device=DEV, generator=g) * 3 + 0.1) \
            + torch.randn(c, device=DEV, generator=g) * 4
        _BnReluFn.apply(y, bn.weight, bn.bias, bn, True)
        assert int(bn.num_batches_tracked) == step
        f = f32(momentum if momentum is not None else 1.0 / step)
        y64 = y.double()
        m, v = y64.mean(0), y64.var(0, unbiased=False)
        unb = v * n / (n - 1)
        vr = var_rel(m, v, L, eps=0.0)
        nm = (1 - f) * rm + f * m
        nv = (1 - f) * rv + f * unb
        bm = (1 - f) * bm + C_RUN * (U * ((1 - f) * rm.abs() + f * m.abs() + nm.abs()) + f * U * m.abs())
        bv = (1 - f) * bv + C_RUN * (U * ((1 - f) * rv.abs() + f * unb + nv.abs()) + f * (U + 4 * vr) * unb)
        rm, rv = nm, nv
        check_elements(capsys, f"running_mean n={n} C={c} momentum={momentum} step {step}", bn.running_mean, rm, bm + TINY)
        check_elements(capsys, f"running_var n={n} C={c} momentum={momentum} step {step}", bn.running_var, rv, bv + TINY)


def bn_bwd_ref(y, gy, out, relu, gamma, mean, invstd, n_total=None):
    N = y.shape[0] if n_total is None else n_total
    gm = gy.double() * ((out > 0).double() if relu else 1.0)
    x = (y.double() - mean.double()) * invstd.double()
    gb, gg = gm.sum(0), (gm * x).sum(0)
    k = (torch.ones_like(gb) if gamma is None else gamma.double()) * invstd.double()
    gx = k * (gm - gb / N - x * gg / N)
    bnd_gx = C_BWD * U * k.abs() * (gm.abs() + gb.abs() / N + x.abs() * (gm * x).abs().sum(0) / N) + TINY
    return gx, gg, gb, bnd_gx, C_BWD * U * (gm * x).abs().sum(0) + TINY, C_BWD * U * gm.abs().sum(0) + TINY


def row_spread_grad(n, c, g, span=30):
    return torch.randn(n, c, device=DEV, generator=g) * torch.exp2(torch.randint(-span, span + 1, (n, 1), device=DEV,
                                                                                 generator=g).float())


@pytest.mark.parametrize("n,c", [(65, 33), (1024, 100), (4097, 2048), (131073, 33)])
@pytest.mark.parametrize("relu", [True, False])
@pytest.mark.parametrize("grad", ["spread", "affine"])
def test_bn_backward_fp64(capsys, n, c, relu, grad):
    """teacher-forced on the kernel's forward; "affine" is g = a + b x (x on the kernel's statistics), where the true gx
    of the un-masked layer is 0"""
    y, gamma, beta, off = bn_inputs(n, c, seed=n + 3 * c)
    out, mean, invstd = ops.bn_relu_forward(y, gamma, beta, None, None, 0.1, EPS, relu)
    g = gen(n * c + 1)
    if grad == "spread":
        gy = row_spread_grad(n, c, g)
    else:
        x = (y.double() - mean.double()) * invstd.double()
        gy = (torch.randn(c, device=DEV, generator=g, dtype=torch.float64) * 2
              + torch.randn(c, device=DEV, generator=g, dtype=torch.float64) * x).float()
    gx, gg, gb = ops.bn_relu_backward(y, gy, out, relu, gamma, mean, invstd)
    gx64, gg64, gb64, bgx, bgg, bgb = bn_bwd_ref(y, gy, out, relu, gamma, mean, invstd)
    name = f"bn bwd {n}x{c} relu={relu} {grad}"
    check_elements(capsys, name + " gx", gx, gx64, bgx)
    check_elements(capsys, name + " g_gamma", gg, gg64, bgg)
    check_elements(capsys, name + " g_beta", gb, gb64, bgb)


# ------------------------------------------------------------------ synchronised BatchNorm on virtual ranks
class VirtualRanks:
    """torch.distributed.all_reduce for ops' `group` branch: `record` keeps each call's tensor, `replay` writes the fp64
    sum of the recorded tensors of the same call index (the same per-rank call order on every virtual rank)"""

    def __init__(self):
        self.recorded, self.total, self.mode = [], None, "record"

    def __call__(self, t, group=None, **kw):
        if self.mode == "record":
            self.recorded.append(t.clone())
        else:
            t.copy_(self.total)

    def replay(self):
        self.total = torch.stack(self.recorded).sum(0)
        self.mode = "replay"


SHARDS = {2: [700, 324], 3: [5, 700, 319], 8: [1, 0, 200, 64, 65, 3, 500, 191]}


@pytest.mark.parametrize("ranks", [2, 3, 8])
@pytest.mark.parametrize("relu", [True, False])
def test_bn_sync_virtual_ranks_fp64(capsys, monkeypatch, ranks, relu):
    import torch.distributed as dist
    c = 100
    sizes = SHARDS[ranks]
    N = sum(sizes)
    y, gamma, beta, off = bn_inputs(N, c, seed=N + ranks)
    y = y[:, (off <= SUPPORTED)]                  # supported range only (every channel asserted)
    c = y.shape[1]
    gamma, beta = gamma[: c], beta[: c]
    parts = list(torch.split(y, sizes))
    rm0, rv0 = torch.randn(c, device=DEV), torch.rand(c, device=DEV) + 0.5
    group = object()

    vr = VirtualRanks()
    monkeypatch.setattr(dist, "all_reduce", vr)
    for p in parts:                                # recording pass: the running statistics of clones move
        ops.bn_relu_forward(p, gamma, beta, rm0.clone(), rv0.clone(), 0.1, EPS, relu, group=group, n_total=N)
    vr.replay()
    res = []
    for p in parts:
        rm, rv = rm0.clone(), rv0.clone()
        out, mean, invstd = ops.bn_relu_forward(p, gamma, beta, rm, rv, 0.1, EPS, relu, group=group, n_total=N)
        res.append((out, mean, invstd, rm, rv))
    for r in res[1:]:                              # every rank holds the same statistics, bit for bit
        for a, b in zip(r[1:], res[0][1:]):
            assert torch.equal(bits(a), bits(b))
    out = torch.cat([r[0] for r in res])
    mean, invstd, rm, rv = res[0][1:]
    L = max(chain(max(s, 1), bn_splits(max(s, 1), c)) for s in sizes) + 16 + ranks
    name = f"bn sync fwd R={ranks} relu={relu}"
    check_bn_forward(capsys, name, y, gamma, beta, relu, out, mean, invstd, L)
    _, m, v, *_ = bn_fwd_ref(y, gamma, beta, relu)
    f = f32(0.1)
    unb = v * N / (N - 1)                          # over the global batch
    rv64 = (1 - f) * rv0.double() + f * unb
    big = rv64 >= 2.0 ** 128                       # the 2^120 channels: beyond fp32, inf as in torch
    assert torch.isinf(rv[big]).all()
    check_elements(capsys, name + " running_var", rv[~big], rv64[~big],
                   (C_RUN * (U * ((1 - f) * rv0.double().abs() + 2 * f * unb) + f * (U + 4 * var_rel(m, v, L)) * unb) + TINY)[~big])
    check_elements(capsys, name + " running_mean", rm, (1 - f) * rm0.double() + f * m,
                   C_RUN * U * ((1 - f) * rm0.double().abs() + 3 * f * m.abs()) + TINY)

    gy = row_spread_grad(N, c, gen(N + 5))
    gparts = list(torch.split(gy, sizes))
    outs = [r[0] for r in res]
    vr = VirtualRanks()
    monkeypatch.setattr(dist, "all_reduce", vr)
    for p, gp, o in zip(parts, gparts, outs):
        ops.bn_relu_backward(p, gp, o, relu, gamma, mean, invstd, group=group, n_total=N)
    vr.replay()
    bw = [ops.bn_relu_backward(p, gp, o, relu, gamma, mean, invstd, group=group, n_total=N)
          for p, gp, o in zip(parts, gparts, outs)]
    gx = torch.cat([b[0] for b in bw])
    gg = torch.stack([b[1] for b in bw]).double().sum(0)     # what the trainer's gradient all-reduce adds up
    gb = torch.stack([b[2] for b in bw]).double().sum(0)
    gx64, gg64, gb64, bgx, bgg, bgb = bn_bwd_ref(y, gy, out, relu, gamma, mean, invstd)
    name = f"bn sync bwd R={ranks} relu={relu}"
    check_elements(capsys, name + " gx", gx, gx64, bgx)
    check_elements(capsys, name + " sum of local g_gamma", gg, gg64, bgg)
    check_elements(capsys, name + " sum of local g_beta", gb, gb64, bgb)


# ------------------------------------------------------------------ exact properties
def bn_both(y, gamma, beta, relu, gy, eps=EPS):
    out, mean, invstd = ops.bn_relu_forward(y, gamma, beta, None, None, 0.1, eps, relu)
    gx, gg, gb = ops.bn_relu_backward(y, gy, out, relu, gamma, mean, invstd)
    return out, mean, invstd, gx, gg, gb


@pytest.mark.parametrize("n,c", [(1024, 100), (4097, 2048), (65, 33)])
@pytest.mark.parametrize("relu", [True, False])
def test_bn_exact_properties(n, c, relu):
    g = gen(n + c + 11)
    y = torch.randn(n, c, device=DEV, generator=g) * 1.7 + 0.3
    gamma, beta = torch.randn(c, device=DEV, generator=g), torch.randn(c, device=DEV, generator=g)
    gy = torch.randn(n, c, device=DEV, generator=g)
    base = bn_both(y, gamma, beta, relu, gy)
    assert all(same_bits(a, b) for a, b in zip(base, bn_both(y, gamma, beta, relu, gy)))          # repeat calls

    perm = torch.randperm(c, device=DEV, generator=g)                                              # column permutation
    pr = bn_both(y[:, perm].contiguous(), gamma[perm], beta[perm], relu, gy[:, perm].contiguous())
    for a, b in zip(base, pr):
        assert same_bits(a[..., perm], b)

    ones, zeros = torch.ones(c, device=DEV), torch.zeros(c, device=DEV)                            # None == ones / zeros
    for a, b in zip(bn_both(y, None, None, relu, gy), bn_both(y, ones, zeros, relu, gy)):
        assert same_bits(a, b)

    e0 = bn_both(y, gamma, beta, relu, gy, eps=0.0)                                                # exact 2^e scaling
    for e in (-40, -17, -1, 1, 9, 40):
        s = 2.0 ** e
        es = bn_both(y * s, gamma, beta, relu, gy, eps=0.0)
        assert same_bits(es[0], e0[0]) and same_bits(es[4], e0[4]) and same_bits(es[5], e0[5]), e
        assert same_bits(es[1], e0[1] * s) and same_bits(es[2], e0[2] / s) and same_bits(es[3], e0[3] / s), e

    yc = y.clone()                                                                                 # constant channels
    yc[:, ::5] = yc[0, ::5]
    oc = ops.bn_relu_forward(yc, gamma, beta, None, None, 0.1, EPS, relu)[0]
    want = beta[::5].clamp_min(0) if relu else beta[::5]
    assert same_bits(oc[:, ::5], want[None, :].expand(n, -1).contiguous())


@pytest.mark.parametrize("poison", [math.nan, math.inf, -math.inf])
@pytest.mark.parametrize("relu", [True, False])
def test_bn_nonfinite_confined_to_channel(poison, relu):
    """torch: mean / var of a channel holding NaN or +-inf are NaN, so the whole channel is; nothing leaks elsewhere"""
    n, c, r, col = 1024, 100, 333, 37
    g = gen(99)
    y = torch.randn(n, c, device=DEV, generator=g) * 1.7 + 0.3
    gamma, beta = torch.rand(c, device=DEV, generator=g) + 0.5, torch.randn(c, device=DEV, generator=g)
    gy = torch.randn(n, c, device=DEV, generator=g)
    clean = bn_both(y, gamma, beta, relu, gy)
    other = torch.arange(c, device=DEV) != col
    yp = y.clone()
    yp[r, col] = poison
    bad = bn_both(yp, gamma, beta, relu, gy)
    assert not torch.isfinite(bad[0][:, col]).any()
    assert not math.isfinite(bad[1][col].item()) and not math.isfinite(bad[2][col].item())
    assert not torch.isfinite(bad[3][:, col]).any() and not math.isfinite(bad[4][col].item())
    for a, b in zip(clean, bad):
        assert same_bits(a[..., other], b[..., other])
    gp = gy.clone()                                                                                # in the gradient
    gp[r, col] = poison
    o, mean, invstd = clean[:3]
    if relu:
        o = o.clone()
        o[r, col] = 1.0                                     # keep the poisoned element inside the ReLU mask
    gx, gg, gb = ops.bn_relu_backward(y, gp, o, relu, gamma, mean, invstd)
    gx0, gg0, gb0 = ops.bn_relu_backward(y, gy, o, relu, gamma, mean, invstd)
    assert not torch.isfinite(gx[:, col]).any() and not math.isfinite(gb[col].item())
    for a, b in zip((gx0, gg0, gb0), (gx, gg, gb)):
        assert same_bits(a[..., other], b[..., other])


def test_bn_batch_of_one_row_raises_like_torch():
    """F.batch_norm refuses a training batch of one row; so do the kernels' autograd node and MLPLayers, on the global
    batch when synchronised"""
    with pytest.raises(ValueError, match="Expected more than 1 value per channel when training"):
        torch.nn.BatchNorm1d(8).to(DEV).train()(torch.randn(1, 8, device=DEV))
    mlp = MLPLayers([16, 8, 4], bn=True).to(DEV).train()
    with pytest.raises(ValueError, match="Expected more than 1 value per channel when training"):
        mlp(torch.randn(1, 16, device=DEV))
    assert mlp(torch.randn(2, 16, device=DEV)).shape == (2, 4)
    bn = torch.nn.BatchNorm1d(8).to(DEV).train()
    bn.lcrec_sync = (object(), 1)
    with pytest.raises(ValueError, match="Expected more than 1 value per channel when training"):
        _BnReluFn.apply(torch.randn(1, 8, device=DEV), bn.weight, bn.bias, bn, True)
    assert int(bn.num_batches_tracked) == 0                 # refused before the running statistics move


# ================================================================== reconstruction loss
def spread_pair(total, seed, span=60):
    """o, x with |elements| = [1, 2) x 2^e, e uniform in [-span, span], random signs"""
    g = gen(seed)

    def one():
        e = torch.randint(-span, span + 1, (total,), device=DEV, generator=g).float()
        s = torch.where(torch.rand(total, device=DEV, generator=g) < 0.5, -1.0, 1.0)
        return s * (torch.rand(total, device=DEV, generator=g) + 1) * torch.exp2(e)
    return one(), one()


def grad_replay(o, x, kind, up):
    inv = np.float32(1.0 / o.numel())
    k = np.float32(np.float32(2.0 if kind == "mse" else 1.0) * inv) * np.float32(1.0 if up is None else up)
    if kind == "mse":
        return torch.tensor(k, device=DEV) * (o - x)
    return torch.tensor(k, device=DEV) * ((o > x).float() - (o < x).float())


LOSS_TOTALS = [1, 2, 3, 5, 4095, 4096, 4097, 1024 * 4096, 4096 * 4096 + 3, 2 * 4096 * 4096 + 5]


@pytest.mark.parametrize("total", LOSS_TOTALS)
@pytest.mark.parametrize("kind", ["mse", "l1"])
def test_recon_loss_fp64(capsys, total, kind):
    o, x = spread_pair(total, seed=total)
    loss = ops.recon_loss(o, x, kind)
    d = o.double() - x.double()
    l64 = (d * d if kind == "mse" else d.abs()).mean()
    check_elements(capsys, f"recon {kind} loss total={total}", loss.reshape(1), l64.reshape(1),
                   (C_LOSS * U * l64 + TINY).reshape(1))
    up = f32(-0.37)
    grad = ops.recon_loss_backward(o, x, kind, torch.tensor(up, device=DEV))
    assert same_bits(grad, grad_replay(o, x, kind, up))
    assert same_bits(ops.recon_loss_backward(o, x, kind, None), ops.recon_loss_backward(o, x, kind, torch.tensor(1.0, device=DEV)))


@pytest.mark.parametrize("kind", ["mse", "l1"])
def test_recon_grad_at_ties_and_nan(kind):
    """o == x gives 0; a NaN difference gives NaN (mse) or 0 (l1, sign(NaN) = 0 as in torch's l1_loss backward)"""
    o, x = spread_pair(4096 * 3 + 2, seed=5, span=4)
    x[::3] = o[::3]
    o[1::7] = math.nan
    grad = ops.recon_loss_backward(o, x, kind, None)
    assert same_bits(grad, grad_replay(o, x, kind, None))
    assert (grad[::3][~torch.isnan(o[::3])] == 0).all()
    if kind == "l1":
        assert (grad[1::7] == 0).all()
        k = f32(1.0 / o.numel())
        assert set(grad.unique().tolist()) <= {-k, 0.0, k}


def offset_copy(t, k):
    """t's values in a flat view starting k floats into a larger buffer (4k bytes past a 16-byte boundary when k < 4)"""
    buf = torch.empty(t.numel() + 4, device=DEV)
    v = buf.view(-1)[k: k + t.numel()]
    v.copy_(t.reshape(-1))
    return v


@pytest.mark.parametrize("total", [5, 4097, 100003])
@pytest.mark.parametrize("kind", ["mse", "l1"])
def test_recon_loss_unaligned_views(total, kind):
    """flat offset views (`view(-1)[k:]`, 4-byte aligned only) give the aligned copy's loss and gradient bit for bit"""
    lib = _lib.load()
    o, x = spread_pair(total, seed=total + 1, span=20)
    loss0 = ops.recon_loss(o, x, kind)
    grad0 = ops.recon_loss_backward(o, x, kind, None)
    for ko, kx, kg in [(1, 1, 0), (2, 0, 3), (0, 3, 1), (3, 2, 2)]:
        ov, xv = offset_copy(o, ko), offset_copy(x, kx)
        assert ov.data_ptr() % 16 == 4 * ko and xv.data_ptr() % 16 == 4 * kx
        assert same_bits(ops.recon_loss(ov, xv, kind), loss0), (ko, kx)
        gv = offset_copy(torch.zeros_like(o), kg)
        with torch.cuda.device(DEV):
            _lib.check(lib.lcrec_recon_loss_backward(C.c_void_p(ov.data_ptr()), C.c_void_p(xv.data_ptr()), total,
                                                     0 if kind == "mse" else 1, C.c_void_p(0), C.c_void_p(gv.data_ptr()),
                                                     C.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)))
        assert same_bits(gv, grad0), (ko, kx, kg)


# ================================================================== fused optimisers
OPT_SIZES = [0, 1, 1023, 1025, 4095, 4096, 4097, 2048 * 4096] + [3, 4, 31, 32, 255, 256, 257, 511, 1000, 2047, 2049, 3000,
                                                                  4098, 5000, 8191, 8192, 8193, 12289, 16384, 20000, 40961,
                                                                  7, 2, 5, 9, 13, 100, 129, 640, 777, 1500, 2500, 3333,
                                                                  6000, 9999, 4096 * 5 - 1, 65537, 33, 65]
ZERO_T = 4                              # tensor whose first 100 gradients (and moments) are zero


def opt_case(seed, nonzero_state):
    """47 parameters; tensor i's gradients randn * 2^e_i, e_i from -40 to 40 over the list (0 at ZERO_T[:100]); moments
    randn-sized at the gradient's scale (m) and its square (v), or zero"""
    assert len(OPT_SIZES) == 47
    g = gen(seed)
    exps = np.round(np.linspace(-40, 40, len(OPT_SIZES))).astype(int)
    order = torch.randperm(len(OPT_SIZES), generator=torch.Generator().manual_seed(seed)).tolist()
    ps, gs, ms, vs = [], [], [], []
    for i, s in enumerate(OPT_SIZES):
        shape = (2048, 4096) if s == 2048 * 4096 else (s,)
        sc = 2.0 ** float(exps[order[i]])
        ps.append(torch.randn(shape, device=DEV, generator=g))
        gs.append(torch.randn(shape, device=DEV, generator=g) * sc)
        ms.append(torch.randn(shape, device=DEV, generator=g) * sc * 0.3 if nonzero_state else torch.zeros(shape, device=DEV))
        vs.append((torch.randn(shape, device=DEV, generator=g) * sc) ** 2 if nonzero_state else torch.zeros(shape, device=DEV))
    gs[ZERO_T].view(-1)[:100] = 0
    ms[ZERO_T].view(-1)[:100] = 0
    vs[ZERO_T].view(-1)[:100] = 0
    return ps, gs, ms, vs


def leaves(ps, gs):
    out = []
    for p, gr in zip(ps, gs):
        q = p.clone().requires_grad_(True)
        q.grad = gr.clone()
        out.append(q)
    return out


def rnd(x):
    """error bound of one fp32 rounding of a result of magnitude |x|"""
    return U * x.abs() + TINY


def sqrt_err(s, es):
    r = torch.sqrt(s)
    return torch.minimum(torch.where(r > 0, es / (2 * r), torch.full_like(r, math.inf)), torch.sqrt(es)) + rnd(r)


def check_clip(capsys, name, gs, gcs, norm, max_norm):
    """total norm against fp64; the written-back gradient == fl(g coef) replayed from the returned norm"""
    n64 = math.sqrt(sum(float((gr.double() ** 2).sum()) for gr in gs))
    nk = float(norm)
    check_elements(capsys, name + " total norm", torch.tensor([nk]), torch.tensor([n64], dtype=torch.float64),
                   torch.tensor([C_NORM * U * n64 + TINY], dtype=torch.float64))
    c = np.float32(max_norm) / (np.float32(nk) + np.float32(1e-6))
    coef = min(np.float32(1.0), c)
    for i, (gr, gc) in enumerate(zip(gs, gcs)):
        assert same_bits(gc, gr * torch.tensor(coef, device=DEV)), (name, i, float(coef))
    return float(coef)


ADAM_CASES = [(True, 1e-2), (False, 1e-2), (True, 0.0)]


@pytest.mark.parametrize("decoupled,wd", ADAM_CASES)
@pytest.mark.parametrize("step", [1, 2, 10000])
@pytest.mark.parametrize("max_norm", [1.0, 2.0 ** 80, 0.0])
def test_adam_fp64(capsys, decoupled, wd, step, max_norm):
    lr, b1, b2, eps = 1e-3, 0.9, 0.999, 1e-8
    ps, gs, ms, vs = opt_case(step + int(decoupled) + int(wd * 100), nonzero_state=step > 1)
    qs = leaves(ps, gs)
    opt = FusedAdam(qs, lr=lr, betas=(b1, b2), eps=eps, weight_decay=wd, decoupled=decoupled)
    for q, m, v in zip(qs, ms, vs):
        opt.state[q].update(step=torch.tensor(float(step - 1)), exp_avg=m.clone(), exp_avg_sq=v.clone())
    norm = opt.clip_and_step(max_norm, want_norm=True)
    name = f"adam{'w' if decoupled else ''} wd={wd} step={step} max_norm={max_norm:g}"
    if max_norm > 0:
        coef = check_clip(capsys, name, gs, [q.grad for q in qs], norm.item(), max_norm)
        report(capsys, name + " clip coefficient", coef, what="value")
    else:
        assert norm is None and all(same_bits(q.grad, gr) for q, gr in zip(qs, gs))
    assert float(opt.state[qs[0]]["step"]) == step
    hyp = (C.c_float * 3)()
    _lib.check(_lib.load().lcrec_adam_hyper(lr, b1, b2, wd, step, hyp))
    decay, step_size, bc2 = (float(h) for h in hyp)
    omb1, omb2, b2f, epsf, wdf = f32(1 - b1), f32(1 - b2), f32(b2), f32(eps), f32(wd)
    worst = {"m": 0.0, "v": 0.0, "p": 0.0}
    for i, (q, p0, m0, v0) in enumerate(zip(qs, ps, ms, vs)):
        if q.numel() == 0:
            continue
        g = q.grad.double()                           # the clipped gradient, teacher-forced
        p, m, v = p0.double(), m0.double(), v0.double()
        if decoupled:
            p1, ep1 = p * decay, rnd(p * decay)
            eg = torch.zeros_like(g)
        else:
            p1, ep1 = p, torch.zeros_like(p)
            if wdf != 0:
                g = g + wdf * p
                eg = rnd(g)
            else:
                eg = torch.zeros_like(g)
        m1 = m + (g - m) * omb1
        em = omb1 * (rnd(g - m) + eg) + rnd(m1)
        v1 = v * b2f + g * g * omb2
        ev = omb2 * (rnd(g * g) + 2 * g.abs() * eg) + rnd(v * b2f) + rnd(v1)
        a = torch.sqrt(v1) / bc2
        ea = sqrt_err(v1, ev) / bc2 + rnd(a)
        den = a + epsf
        eden = ea + rnd(den)
        qv = m1 / den
        eq = em / den + qv.abs() * eden / den + rnd(qv)
        p2 = p1 - step_size * qv
        ep = ep1 + step_size * eq + rnd(p2)
        st = opt.state[q]
        worst["m"] = max(worst["m"], check_elements(capsys, f"{name} t{i} m", st["exp_avg"], m1, C_OPT * em, show=False))
        worst["v"] = max(worst["v"], check_elements(capsys, f"{name} t{i} v", st["exp_avg_sq"], v1, C_OPT * ev, show=False))
        worst["p"] = max(worst["p"], check_elements(capsys, f"{name} t{i} p", q.detach(), p2, C_OPT * ep, show=False))
    for k, r in worst.items():
        report(capsys, f"{name} all tensors {k}", r)
    if wd == 0:                                       # g = 0 with v = 0: p exactly unchanged
        assert same_bits(qs[ZERO_T].detach().view(-1)[:100], ps[ZERO_T].view(-1)[:100])


@pytest.mark.parametrize("step", [1, 10000])
@pytest.mark.parametrize("max_norm", [1.0, 0.0])
def test_adam_device_hyper_equals_host(step, max_norm):
    ps, gs, ms, vs = opt_case(77 + step, nonzero_state=step > 1)
    runs = []
    for dev in (False, True):
        qs = leaves(ps, gs)
        opt = FusedAdam(qs, lr=1e-3, weight_decay=1e-2)
        for q, m, v in zip(qs, ms, vs):
            opt.state[q].update(step=torch.tensor(float(step - 1)), exp_avg=m.clone(), exp_avg_sq=v.clone())
        if dev:
            opt.prepare_hyper()
        norm = opt.clip_and_step(max_norm, want_norm=True, device_hyper=dev)
        runs.append((qs, opt, norm))
    (qa, oa, na), (qb, ob, nb) = runs
    assert (na is None) == (nb is None) and (na is None or same_bits(na, nb))
    for a, b in zip(qa, qb):
        assert same_bits(a.detach(), b.detach()) and same_bits(a.grad, b.grad)
        assert same_bits(oa.state[a]["exp_avg"], ob.state[b]["exp_avg"])
        assert same_bits(oa.state[a]["exp_avg_sq"], ob.state[b]["exp_avg_sq"])


@pytest.mark.parametrize("kind", ["sgd", "adagrad", "rmsprop"])
@pytest.mark.parametrize("wd", [1e-2, 0.0])
@pytest.mark.parametrize("max_norm", [1.0, 0.0])
def test_simple_optimisers_fp64(capsys, kind, wd, max_norm):
    lr = 1e-2
    ps, gs, ms, vs = opt_case(200 + len(kind), nonzero_state=True)
    qs = leaves(ps, gs)
    opt = FusedSimple(qs, kind, lr=lr, weight_decay=wd)
    key = {"sgd": None, "adagrad": "sum", "rmsprop": "square_avg"}[kind]
    if key:
        for q, v in zip(qs, vs):
            opt.state[q].update(step=torch.tensor(3.0), **{key: v.clone()})
    opt.clip_and_step(max_norm)
    name = f"{kind} wd={wd} max_norm={max_norm:g}"
    if max_norm <= 0:
        assert all(same_bits(q.grad, gr) for q, gr in zip(qs, gs))
    group = opt.param_groups[0]
    lrf, wdf, epsf = f32(lr), f32(wd), f32(group.get("eps", 0.0))
    alpha, oma = f32(group.get("alpha", 0.99)), f32(1 - group.get("alpha", 0.99))
    worst = {"s": 0.0, "p": 0.0}
    for i, (q, p0, s0) in enumerate(zip(qs, ps, vs)):
        if q.numel() == 0:
            continue
        g, p, s = q.grad.double(), p0.double(), s0.double()
        if wdf != 0:
            g = g + wdf * p
            eg = rnd(g)
        else:
            eg = torch.zeros_like(g)
        if kind == "sgd":
            p2 = p - lrf * g
            ep = lrf * eg + rnd(p2)
        else:
            if kind == "adagrad":
                s1 = s + g * g
                es = 2 * g.abs() * eg + rnd(s1)
            else:
                s1 = s * alpha + g * g * oma
                es = oma * (rnd(g * g) + 2 * g.abs() * eg) + rnd(s * alpha) + rnd(s1)
            worst["s"] = max(worst["s"], check_elements(capsys, f"{name} t{i} state", opt.state[q][key], s1, C_OPT * es, show=False))
            r = torch.sqrt(s1)
            den = r + epsf
            eden = sqrt_err(s1, es) + rnd(den)
            qv = g / den
            eq = eg / den + qv.abs() * eden / den + rnd(qv)
            p2 = p - lrf * qv
            ep = lrf * eq + rnd(p2)
        worst["p"] = max(worst["p"], check_elements(capsys, f"{name} t{i} p", q.detach(), p2, C_OPT * ep, show=False))
    for k, r in worst.items():
        report(capsys, f"{name} all tensors {k}", r)


def test_simple_clip_replay(capsys):
    """the simple optimisers' clip prologue: norm against fp64 and the written-back fl(g coef), bit for bit"""
    ps, gs, ms, vs = opt_case(300, nonzero_state=False)
    for kind in ("sgd", "adagrad", "rmsprop"):
        qs = leaves(ps, gs)
        FusedSimple(qs, kind, lr=1e-2).clip_and_step(1.0)
        # FusedSimple does not return the norm: recover it from the Adam kernel's identical pass 1
        qa = leaves(ps, gs)
        norm = FusedAdam(qa, lr=0.0).clip_and_step(1.0, want_norm=True)
        check_clip(capsys, f"{kind} clip", gs, [q.grad for q in qs], norm.item(), 1.0)


@pytest.mark.parametrize("kind", ["adamw", "adam", "sgd", "adagrad", "rmsprop"])
def test_nan_gradient_poisons_every_parameter(kind):
    """clip_grad_norm_ + step in torch: a NaN gradient makes the total norm and so every clipped gradient NaN"""
    ps, gs, ms, vs = opt_case(400, nonzero_state=False)
    gs[10].view(-1)[3] = math.nan
    qs = leaves(ps, gs)
    if kind.startswith("adam"):
        FusedAdam(qs, lr=1e-3, weight_decay=1e-2, decoupled=kind == "adamw").clip_and_step(1.0)
    else:
        FusedSimple(qs, kind, lr=1e-2).clip_and_step(1.0)
    for q in qs:
        assert torch.isnan(q.detach()).all()
