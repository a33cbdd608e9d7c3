"""Encoder GEMMs element by element against fp64 (B200).

Every value the split-operand kernels write is compared with a plain float64 evaluation of the same operation, with a
bound per element instead of a global mean:

    |y - y64| <= C * (|a| @ |W|^T + |b|) + FLOOR * ([a != 0] G_a @ |W|^T + |a| @ ([w != 0] G_w)^T) + 2^-148

The first term is the fp32-level error of the two-term operand split and of the fp32 accumulation.  The second is the
representation floor of the design: an fp16 hi/lo pair scaled to [2^14, 2^15) keeps a value to a fixed fraction of its
scale group's maximum (G_a = max |a| over the element's scale group: 256 columns of a row on the CTA-pair path, the
whole row on the single-CTA path; G_w = max |w| of the output channel; no floor on the tf32 engine).  Exact zeros split
exactly and carry no floor, so an output that reads a single small scale group is held to that group's maximum, not to
the row's.  The last term
is the resolution of fp32 subnormals.  Inputs are built where kernels go wrong: scale groups of one row 2^80 apart,
zero rows and groups, groups with one non-zero element, output channels that read a single scale group, ReLU-zeroed
hidden groups, tile column halves 2^10 apart, same-sign operands, ragged shapes, and a magnitude sweep over the whole
fp32 range.  Exact properties (power-of-two row scaling, row permutation and subsets, `want_acts`, non-finite rows)
are asserted bit for bit.  The worst ratio |y - y64| / bound of each case is printed."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from lcrec_b200 import ops
    DEV = torch.device("cuda:0")

# Per-element constants (C of the module docstring), about 4x the worst ratio measured on a B200 (DESIGN.md section 4.1).
C_MIXED = 2e-6         # operands of both signs (measured 8.9e-7)
C_SAME_SIGN = 1e-5     # x >= 0, W >= 0: the truncating TMEM accumulator's bias is not cancelled (measured 2.6e-6)
C_BWD = 1e-5           # gradient GEMMs: items 2^16 apart leave a few dominant terms per sum, whose truncation errors do
                       # not average out (measured 2.5e-6)
C_GB = 1e-6            # bias gradient, per column, against sum |g| (measured 1.4e-7)
FLOOR = 2.0 ** -37     # 4x the 2^-39 representation floor (the MMA keeps fp16 subnormals; measured 2^-42)
TINY = 2.0 ** -148     # two fp32 subnormal steps

RUNSH = [4096, 2048, 1024, 512, 256, 128, 64, 32]
ARCHS = {
    "runsh": RUNSH,                            # pair kernel, 128 / 64 narrow pair tiles, single-CTA 64 -> 32
    "single_first": [200, 96, 512, 256, 32],   # split_f16_rows layer, then split_groups into pair layers
    "ragged": [4104, 512, 128, 64, 16],        # k % 256 == 8: a ragged last scale group on the pair kernel
    "odd_k": [300, 256, 48, 12],               # k not a multiple of 8 (300), k = 48 < 64 on the single-CTA kernel
    "small": [96, 64, 48, 16],                 # the small model
}
# (engine, set_variant): f16 x3 default, f16 x3 without the pair kernel, pair kernel with 6 x 32 KB stages, tf32 x3
CFGS = {"e1": (1, 0), "e1_nopair": (1, 16), "e1_stage6": (1, 32), "e0": (0, 0)}
ROWS_RUNSH = [1, 127, 128, 129, 255, 256, 257, 4097, 131073]


def report(capsys, name, ratio):
    with capsys.disabled():
        print(f"\n  [{name}] worst |y - y64| / bound = {ratio:.3e}")


def gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def pair_served(engine, variant, k, n_out):
    """linear_pair_supported of csrc/linear_pair.cu, as MlpHandle routes a layer"""
    return (engine == 1 and not (variant & 16) and (n_out % 256 == 0 or n_out in (128, 64)) and k >= 64
            and k % 8 == 0)


def group_max(a, group):
    """max |a| over each element's scale group of `group` columns (None: whole row) -> same shape, fp64"""
    a = a.abs().double()
    if group is None or group >= a.shape[1]:
        return a.amax(1, keepdim=True).expand_as(a)
    rows, k = a.shape
    pad = (-k) % group
    g = torch.nn.functional.pad(a, (0, pad)).view(rows, -1, group).amax(2, keepdim=True)
    return g.expand(-1, -1, group).reshape(rows, -1)[:, :k]


def gemm_bound(a, w, b, c, group_a, split_w=True):
    """(y64, bound) of a @ w^T + b for fp32 a (n, k), w (m, k): group_a = the A scale group (256 / None = row / 0 =
    tf32 engine, no floor); split_w: W carries one scale per output channel (f16 x3 engines)."""
    a64, w64 = a.double(), w.double()
    y64 = a64 @ w64.t()
    if b is not None:
        y64 = y64 + b.double()
    aa, wa = a64.abs(), w64.abs()
    bnd = aa @ wa.t()
    if b is not None:
        bnd = bnd + b.double().abs()
    bnd = c * bnd + TINY
    if group_a != 0:
        bnd = bnd + FLOOR * ((group_max(a, group_a) * (a != 0)) @ wa.t())
        if split_w:
            bnd = bnd + FLOOR * (aa @ (group_max(w, None) * (w != 0)).t())
    return y64, bnd


def check_elements(y, y64, bnd, what):
    """|y - y64| <= bnd everywhere; returns the worst ratio"""
    err = (y.double() - y64).abs()
    bad = ~(err <= bnd)
    if bad.any():
        i = bad.nonzero()[0].tolist()
        raise AssertionError(f"{what}: {int(bad.sum())} elements over the bound, first {i}: y={y[tuple(i)].item()!r} "
                             f"y64={y64[tuple(i)].item()!r} bound={bnd[tuple(i)].item()!r}")
    return (err / bnd).max().item()


def channel_scale(w, engine):
    """the per-output-channel power of two the accumulator carries: 2^15 / max|w_c| (floor) on the f16 engine"""
    if engine == 0:
        return torch.ones(w.shape[0], dtype=torch.float64, device=DEV)
    e = torch.frexp(w.abs().amax(1)).exponent.double()
    return torch.exp2((15 - e).clamp(-126, 126))


# ------------------------------------------------------------------ operands
def hetero_rows(n, k, seed, span=40):
    """randn rows with every (row, 256-column group) scaled by its own power of two in [2^-span, 2^span], plus a zero
    row, a row with an all-zero group, and a row whose first group holds a single non-zero element"""
    g = gen(seed)
    x = torch.randn(n, k, device=DEV, generator=g)
    ng = (k + 255) // 256
    e = torch.randint(-span, span + 1, (n, ng), device=DEV, generator=g).float()
    x *= torch.exp2(e).repeat_interleave(256, 1)[:, :k]
    if n >= 4:
        x[1] = 0
        x[2, : min(k, 256)] = 0
        x[3, 1: min(k, 256)] = 0
    return x


def hostile_weights(dims, seed):
    """W = randn / sqrt(k) with the two column halves of each tile 2^10 apart (2^-5 / 2^5 per output channel), every
    8th channel reading a single 256-column scale group, and (hidden layers of >= 512 channels) channels 256-511 behind
    a bias of -2^100, so that the ReLU zeroes a whole scale group of the next layer's input"""
    g = gen(seed)
    ws, bs = [], []
    for l, (k, m) in enumerate(zip(dims[:-1], dims[1:])):
        w = torch.randn(m, k, device=DEV, generator=g) / math.sqrt(k)
        tile = 256 if m % 256 == 0 else m
        c = torch.arange(m, device=DEV)
        w *= torch.where((c % tile) < tile // 2, 2.0 ** -5, 2.0 ** 5)[:, None]
        ng = (k + 255) // 256
        for ch in range(0, m, 8):
            keep = (ch // 8) % ng
            w[ch, : keep * 256] = 0
            w[ch, (keep + 1) * 256:] = 0
        b = torch.randn(m, device=DEV, generator=g) * 0.01
        b[::8] = 0                             # a bias would hide the single group's contribution below its ulp
        if l < len(dims) - 2 and m >= 512:
            b[256:512] = -2.0 ** 100
        ws.append(w)
        bs.append(b)
    return ws, bs


def plain_weights(dims, seed, same_sign=False, zero_bias=False):
    g = gen(seed)
    ws, bs = [], []
    for k, m in zip(dims[:-1], dims[1:]):
        w = torch.randn(m, k, device=DEV, generator=g) / math.sqrt(k)
        b = torch.randn(m, device=DEV, generator=g) * 0.01
        if same_sign:
            w, b = w.abs(), b.abs()
        ws.append(w)
        bs.append(torch.zeros_like(b) if zero_bias else b)
    return ws, bs


def handle(ws, bs, cfg):
    engine, variant = CFGS[cfg]
    h = ops.MlpHandle(ws, bs)
    h.set_engine(engine)
    h.set_variant(variant)
    return h


def teacher_forced(h, ws, bs, x, cfg, c):
    """forward(x, want_acts=True); every layer against fp64 on the kernel's own previous activation -> worst ratio.
    Channels behind a bias of -2^100 (hostile_weights) must come out exactly 0."""
    engine, variant = CFGS[cfg]
    y, acts = h.forward(x, want_acts=True)
    assert torch.equal(acts[-1], y)
    worst = 0.0
    a = x
    for l, (w, b) in enumerate(zip(ws, bs)):
        k, m = w.shape[1], w.shape[0]
        grp = 0 if engine == 0 else (256 if pair_served(engine, variant, k, m) else None)
        y64, bnd = gemm_bound(a, w, b, c, grp, split_w=engine == 1)
        if l < len(ws) - 1:
            y64 = torch.relu(y64)
            dead = b == -2.0 ** 100
            assert not dead.any() or (acts[l][:, dead] == 0).all(), f"layer {l}: a channel behind -2^100 is not 0"
        worst = max(worst, check_elements(acts[l], y64, bnd, f"layer {l} ({k}->{m})"))
        del y64, bnd
        a = acts[l]
    return worst


# ------------------------------------------------------------------ 1. per-element forward bound, layer by layer
FWD_CASES = [("runsh", n, "e1") for n in ROWS_RUNSH] + [("runsh", n, c) for n in (129, 4097) for c in ("e1_nopair", "e1_stage6", "e0")]
FWD_CASES += [(a, n, c) for a in ARCHS if a != "runsh" for n in (1, 129, 4097) for c in CFGS]


@pytest.mark.parametrize("arch,n,cfg", FWD_CASES)
def test_forward_per_element_bound(arch, n, cfg, capsys):
    dims = ARCHS[arch]
    ws, bs = hostile_weights(dims, seed=len(dims) * 100 + dims[0])
    h = handle(ws, bs, cfg)
    x = hetero_rows(n, dims[0], seed=n + dims[0])
    worst = teacher_forced(h, ws, bs, x, cfg, C_MIXED)
    report(capsys, f"{arch} n={n} {cfg}", worst)


@pytest.mark.parametrize("arch", list(ARCHS))
@pytest.mark.parametrize("cfg", list(CFGS))
def test_forward_same_sign_bound(arch, cfg, capsys):
    """x >= 0, W >= 0, b >= 0 through the whole stack: no cancellation hides the accumulator's truncation bias"""
    dims = ARCHS[arch]
    ws, bs = plain_weights(dims, seed=dims[0] + 1, same_sign=True)
    h = handle(ws, bs, cfg)
    x = torch.randn(4097, dims[0], device=DEV, generator=gen(dims[0])).abs()
    worst = teacher_forced(h, ws, bs, x, cfg, C_SAME_SIGN)
    report(capsys, f"same sign {arch} {cfg}", worst)


LIN_SHAPES = [(4097, 4096, 2048), (257, 4104, 256), (129, 300, 256), (255, 36, 64), (131073, 256, 128), (1000, 512, 64)]


@pytest.mark.parametrize("n,k,m", LIN_SHAPES)
@pytest.mark.parametrize("relu", [True, False])
def test_linear_forward_variants_per_element(n, k, m, relu, capsys):
    """ops.linear_forward: tf32 x3 (0, 1), f16 x3 single CTA (2, 3), CTA pair (6, 7) where the shape allows"""
    ws, bs = hostile_weights([k, m], seed=k + m)
    w, b = ws[0], bs[0]
    x = hetero_rows(n, k, seed=n * 3 + k)
    variants = [0, 1, 2, 3] + ([6, 7] if pair_served(1, 0, k, m) else [])
    worst = 0.0
    for v in variants:
        y = ops.linear_forward(x, w, b, relu, variant=v)
        grp = 0 if v < 2 else (256 if v >= 6 else None)
        y64, bnd = gemm_bound(x, w, b, C_MIXED, grp, split_w=v >= 2)
        if relu:
            y64 = torch.relu(y64)
        worst = max(worst, check_elements(y, y64, bnd, f"variant {v}"))
    report(capsys, f"linear n={n} k={k} m={m} relu={relu}", worst)


# ------------------------------------------------------------------ 2. exact invariances
@pytest.mark.parametrize("arch", ["runsh", "single_first", "small"])
@pytest.mark.parametrize("cfg", ["e1", "e1_nopair", "e0"])
def test_power_of_two_row_scaling_is_exact(arch, cfg):
    """y(diag(2^e) x) == diag(2^e) y(x) bit for bit (zero biases): every scale is a power of two and ReLU is positively
    homogeneous, so this pins each scale index, layout and fold without a tolerance"""
    dims = ARCHS[arch]
    ws, bs = plain_weights(dims, seed=7, zero_bias=True)
    h = handle(ws, bs, cfg)
    n = 4097
    g = gen(11)
    x = torch.randn(n, dims[0], device=DEV, generator=g)
    e = torch.randint(-60, 61, (n, 1), device=DEV, generator=g).float()
    e[0], e[1], e[2] = -60, 60, 0
    y = h.forward(x)
    ys = h.forward(x * torch.exp2(e))
    assert torch.isfinite(y).all()
    assert torch.equal(ys, y * torch.exp2(e))


@pytest.mark.parametrize("cfg", ["e1", "e0"])
def test_rows_are_independent(cfg):
    """y(x[P]) == y(x)[P] and y(x[a:b]) == y(x)[a:b] across tile edges and the 131072-row boundary; forward with
    want_acts returns the same y as without"""
    ws, bs = hostile_weights(RUNSH, seed=5)
    h = handle(ws, bs, cfg)
    n = 131200
    x = hetero_rows(n, RUNSH[0], seed=21)
    y = h.forward(x)
    y2, acts = h.forward(x, want_acts=True)
    assert torch.equal(y2, y)
    p = torch.randperm(n, device=DEV, generator=gen(3))
    assert torch.equal(h.forward(x[p]), y[p])
    for a, b in ((0, 1), (1, 2), (127, 385), (255, 257), (5, 131100), (131071, 131073), (131072, 131200)):
        assert torch.equal(h.forward(x[a:b]), y[a:b]), (a, b)
        ys, acts_s = h.forward(x[a:b], want_acts=True)
        assert torch.equal(ys, y[a:b]) and torch.equal(acts_s[0], acts[0][a:b]), (a, b)


@pytest.mark.parametrize("arch", ["runsh", "single_first", "small"])
@pytest.mark.parametrize("cfg", ["e1", "e1_nopair", "e0"])
def test_non_finite_input_stays_in_its_row(arch, cfg):
    """a row with a NaN, +inf or -inf comes out non-finite wherever the fp64 evaluation does; every other row is
    bit-identical to the clean run (the fused ReLU lets NaN through like torch.relu)"""
    dims = ARCHS[arch]
    ws, bs = plain_weights(dims, seed=9)
    h = handle(ws, bs, cfg)
    n, k = 300, dims[0]
    x = torch.randn(n, k, device=DEV, generator=gen(13))
    clean = h.forward(x)
    bad = {5: (3, float("nan")), 17: (k // 2, float("inf")), 18: (k - 1, float("-inf")), 200: (k - 1, float("nan")),
           256: (0, float("inf"))}
    xb = x.clone()
    for r, (c, v) in bad.items():
        xb[r, c] = v
    got = h.forward(xb)
    rows = torch.tensor(sorted(bad), device=DEV)
    keep = torch.ones(n, dtype=torch.bool, device=DEV)
    keep[rows] = False
    assert torch.equal(got[keep], clean[keep])
    a = xb[rows].double()
    for l, (w, b) in enumerate(zip(ws, bs)):
        a = a @ w.double().t() + b.double()
        if l < len(ws) - 1:
            a = torch.relu(a)
    nonfinite64 = ~torch.isfinite(a)
    assert nonfinite64.any(1).all()
    assert (~torch.isfinite(got[rows]))[nonfinite64].all()


# ------------------------------------------------------------------ 3. magnitude range
def sweep_rows(k, exps, seed, zero_col0=False):
    """row i: every 256-column group of randn scaled so that its maximum is exactly 2^exps[i]"""
    x = torch.randn(len(exps), k, device=DEV, generator=gen(seed))
    if zero_col0:
        x[:, 0] = 0
    gm = group_max(x, 256).float()
    e = torch.tensor(exps, device=DEV, dtype=torch.float32)[:, None]
    return (x / gm) * torch.exp2(e)


def check_range(h, ws, x, cfg, what, capsys):
    """teacher-forced per-element bound wherever |a| @ |W|^T * (channel scale) < 2^127 (the accumulator's range);
    beyond it the output is within the bound or non-finite, and non-finite wherever |y64| * (channel scale) >= 2^128"""
    engine, variant = CFGS[cfg]
    y, acts = h.forward(x, want_acts=True)
    a = x
    worst = 0.0
    for l, w in enumerate(ws):
        k, m = w.shape[1], w.shape[0]
        grp = 0 if engine == 0 else (256 if pair_served(engine, variant, k, m) else None)
        y64, bnd = gemm_bound(a, w, None, C_MIXED, grp, split_w=engine == 1)
        if l < len(ws) - 1:
            y64 = torch.relu(y64)
        out = acts[l]
        fin_in = torch.isfinite(a).all(1, keepdim=True)
        sc = channel_scale(w, engine)[None, :]
        absprod = a.double().abs() @ w.double().abs().t()
        supported = fin_in & (absprod * sc < 2.0 ** 127)
        err = (out.double() - y64).abs()
        within = err <= bnd
        wrong = (supported & ~within) | (~supported & torch.isfinite(out) & ~within)
        if wrong.any():
            i = wrong.nonzero()[0].tolist()
            raise AssertionError(f"{what} layer {l}: {int(wrong.sum())} wrong elements, first {i}: row max "
                                 f"{a[i[0]].abs().max().item()!r} y={out[tuple(i)].item()!r} y64={y64[tuple(i)].item()!r}")
        must_inf = ~fin_in | ~torch.isfinite(y64) | (y64.abs() * sc >= 2.0 ** 128)
        assert not torch.isfinite(out[must_inf]).any(), f"{what} layer {l}: finite output beyond the accumulator range"
        if supported.any():
            worst = max(worst, (err / bnd)[supported].max().item())
        a = out
    report(capsys, what, worst)
    return acts


# smallest input group maximum (power of two) each engine keeps at fp32 accuracy.  The f16 x3 splits scale by at most
# 2^126 (2^-126 would be the smallest normal 1/s): a group maximum below 2^-111 lands in [1, 2^14) instead of
# [2^14, 2^15), and its lo terms are fp16 subnormals, which the MMA keeps.  The tf32 x3 engine has no scales: below
# 2^-114 its lo terms and cross products turn into fp32 subnormals (measured err / (|a| |W|): 1.8e-7 at 2^-114,
# 5.5e-6 at 2^-120, 3.7e-4 at 2^-126; DESIGN.md section 4.1)
SWEEP_FROM = {"e1": -126, "e1_nopair": -126, "e0": -114}


@pytest.mark.parametrize("cfg", ["e1", "e1_nopair", "e0"])
def test_group_maxima_over_the_fp32_range(cfg, capsys):
    """input group maxima 2^-126 ... 2^127 through a pair -> pair -> narrow-pair stack (split_groups, the pair
    epilogue's hand-over, or split_f16_rows on every layer without the pair kernel): never a wrong finite number"""
    dims = [512, 512, 256, 128]
    ws, _ = plain_weights(dims, seed=17, zero_bias=True)
    h = handle(ws, [None] * len(ws), cfg)
    exps = list(range(SWEEP_FROM[cfg], 128))
    x = sweep_rows(dims[0], exps, seed=19)
    acts = check_range(h, ws, x, cfg, f"sweep {cfg}", capsys)
    # the supported range is not empty at either end: the smallest and a large row come out finite
    assert torch.isfinite(acts[-1][0]).all() and torch.isfinite(acts[-1][exps.index(100)]).all()
    if CFGS[cfg][0] == 1:
        # the accumulator carries 2^15 / max|w_c| (2^17 here): 2^127 groups overflow it on every channel
        assert not torch.isfinite(acts[0][-1]).any()


@pytest.mark.parametrize("cfg", ["e1", "e1_nopair"])
def test_huge_groups_with_a_dominant_weight_column(cfg, capsys):
    """group maxima up to 2^127 where the weights are 2^-20 of each channel's maximum: the accumulator stays in range,
    so the operand split itself must not overflow (fp16 hi of x * 2^-100 is inf from 65520 * 2^100 on)"""
    k, m = 512, 256
    w = torch.randn(m, k, device=DEV, generator=gen(23)) * 2.0 ** -20
    w[:, 0] = 1.0
    h = handle([w], [None], cfg)
    exps = list(range(100, 128))
    x = sweep_rows(k, exps, seed=29, zero_col0=True)
    acts = check_range(h, [w], x, cfg, f"dominant column {cfg}", capsys)
    assert torch.isfinite(acts[0]).all()


# ------------------------------------------------------------------ 4. backward against fp64
BWD_N = [1, 7, 37, 255, 256, 1000, 1024, 4097]


def item_scaled(n, k, seed):
    g = gen(seed)
    x = torch.randn(n, k, device=DEV, generator=g)
    return x * torch.exp2(torch.randint(-8, 9, (n, 1), device=DEV, generator=g).float())


def floors(a, w, group_a):
    """the representation-floor (and subnormal) terms of gemm_bound alone"""
    return gemm_bound(a, w, None, 0.0, group_a)[1]


@pytest.mark.parametrize("n", BWD_N)
@pytest.mark.parametrize("k,m", [(512, 256), (96, 64), (1024, 2048)])
def test_linear_backward_per_element(n, k, m, capsys):
    """gx = g W against |g| |W|, gw = g^T x against |g|^T |x| per element, gb against sum |g| per column; item and
    gradient rows 2^-8 ... 2^8 apart within the batch (gw's per-feature scale spans the whole batch).  Batch sizes not
    a multiple of 8 (zero-padded transposes), ragged 256-item groups, gw on and off the pair kernel."""
    ws, bs = plain_weights([k, m], seed=k + m)
    w, b = ws[0], bs[0]
    x = item_scaled(n, k, seed=n + 1)
    gy = item_scaled(n, m, seed=n + 2)
    y = ops.linear_forward(x, w, b, True)
    gx, gw, gb = ops.linear_backward(x, w, y, gy)
    gd = gy * (y > 0).float()
    nr = (n + 7) // 8 * 8
    gx64, bx = gemm_bound(gd, w.t(), None, C_BWD, 256 if pair_served(1, 0, m, k) else None)
    worst = check_elements(gx, gx64, bx, "gx")
    gw64, bw = gemm_bound(gd.t(), x.t(), None, C_BWD, 256 if pair_served(1, 0, nr, k) else None)
    worst = max(worst, check_elements(gw, gw64, bw, "gw"))
    worst_b = check_elements(gb, gd.double().sum(0), C_GB * gd.double().abs().sum(0) + TINY, "gb")
    report(capsys, f"linear_backward n={n} k={k} m={m}", worst)
    report(capsys, f"linear_backward gb n={n} k={k} m={m}", worst_b)


@pytest.mark.parametrize("arch", ["runsh", "single_first", "small"])
@pytest.mark.parametrize("n", [1, 37, 1024, 4097])
def test_mlp_backward_against_fp64_chain(arch, n, capsys):
    """MlpHandle.backward against an fp64 chain through the kernel's own ReLU masks (acts > 0).  The bound is the same
    chain on absolute values with C_BWD per layer passed, plus each layer's representation floors carried down the
    chain (F)."""
    dims = ARCHS[arch]
    ws, bs = plain_weights(dims, seed=31)
    h = handle(ws, bs, "e1")
    x = item_scaled(n, dims[0], seed=n + 5)
    gy = item_scaled(n, dims[-1], seed=n + 6)
    y, acts = h.forward(x, want_acts=True)
    gx, gws, gbs = h.backward(x, acts, gy)
    g64, gabs = gy.double(), gy.double().abs()
    F = torch.zeros_like(g64)
    worst = 0.0
    L = len(ws)
    nr = (n + 7) // 8 * 8
    for l in range(L - 1, -1, -1):
        k, m = dims[l], dims[l + 1]
        if l < L - 1:
            mask = (acts[l] > 0).double()
            g64, gabs, F = g64 * mask, gabs * mask, F * mask
        a = (x if l == 0 else acts[l - 1]).double()
        c = C_BWD * (L - l)
        bw = c * (gabs.t() @ a.abs()) + F.t() @ a.abs() + floors(gabs.t(), a.t(), 256 if pair_served(1, 0, nr, k) else None)
        worst = max(worst, check_elements(gws[l], g64.t() @ a, bw, f"gw[{l}]"))
        worst = max(worst, check_elements(gbs[l], g64.sum(0), (c + C_GB) * gabs.sum(0) + F.sum(0) + TINY, f"gb[{l}]"))
        w64 = ws[l].double()
        F = F @ w64.abs() + floors(gabs, ws[l].t(), 256 if pair_served(1, 0, m, k) else None)
        g64, gabs = g64 @ w64, gabs @ w64.abs()
    worst = max(worst, check_elements(gx, g64, C_BWD * (L + 1) * gabs + F, "gx"))
    report(capsys, f"mlp_backward {arch} n={n}", worst)
