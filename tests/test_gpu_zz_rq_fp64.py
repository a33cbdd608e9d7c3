"""Residual quantiser row by row against fp64 (B200), on every kernel path of `rq_quantize_select`.

Every case is teacher-forced on the kernel's own codes.  The residual entering each level is rebuilt from those codes
with the reference's fp32 operations (`t = q - r; x_res = r + t; r = r - x_res; x_q = x_q + x_res`: IEEE adds with
nothing to contract), so the returned `resid` and `x_q` must equal the replay bit for bit on every row, whatever code
was picked.  On the replayed residual r entering level l the pick must be near-optimal in fp64:

    d64[pick] <= min_k (d64[k] + B[k]) + B[pick],     d64[k] = |r - c_k|^2

    B[k] = C * (|r| + |c_k|)^2                                                       SIMT paths, C = C_SIMT (D + 3) 2^-24
    B[k] = C_TC * (|r| + |c_k|)^2 + FLOOR * (G_r . |c_k| + |r|_1 G_c) + TINY          tensor-core paths

(|r|^2 + |c_k|^2 + 2 |r||c_k| = (|r| + |c_k|)^2.)  Any kernel whose computed distances are within B of the truth
passes, whatever its summation order and tie behaviour, so the window is valid on both paths and on near-ties.
(D + 3) 2^-24 is the worst-case constant of the SIMT evaluation (three length-D fp32 chains, one add, one subtract);
C_SIMT is a fraction of it.  On the tensor-core paths G_r is |r|'s maximum over each element's 256-column scale group
(zero elements split exactly and carry no floor) and G_c the code row's maximum: the representation floor of the
scaled fp16 hi/lo operands, as in tests/test_gpu_zz_encoder_fp64.py.  The window must also have power: on random
data fewer than POWER_MAX of the rows may hold a second code inside it.

sq_err is the fp64 sum of the replayed fl(t * t) to 1e-12.  Exact duplicate codes never lose to their higher copy and
duplicate rows get identical codes and residuals on every path; the SMEM kernels (1, 2 and 4 items per thread, TRAIN)
and the tensor-core path (row permutation, subsets) give bit-identical rows; power-of-two scaling of latents and
codebooks scales the residuals exactly and keeps the codes.  The training forward / backward (rq_train.cu, segsum.cuh)
is checked bit for bit against sequential replays.  Each case prints the path it asserts, its worst window ratio
max_k (d64[pick] - d64[k]) / (B[k] + B[pick]) (<= 1 passes) and its ambiguous-row fraction."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from lcrec_b200 import ops
    DEV = torch.device("cuda:0")

U = 2.0 ** -24
# Window constants (B of the module docstring), about 4x the worst ratio measured on a B200 (DESIGN.md sections 2.2, 4.2).
C_SIMT = 0.65          # fraction of the worst-case (D + 3) 2^-24 of the SIMT kernels and vq_distances (measured 0.166:
                       # vq_distances on rows of 2^-56 .. 2^56 against codes 2^+-20 apart; picks 0.081)
C_TC = 3e-7            # tensor-core paths, relative to (|r| + |c_k|)^2 (measured 7.4e-8 = 1.2 * 2^-24: near-tie picks)
FLOOR = 2.0 ** -37     # representation floor of the scaled fp16 hi/lo pair: the encoder file's constant for the same
                       # split (no case here comes near it)
TINY = 2.0 ** -140     # fp32 subnormal products of tiny rows (D * 2^-149 for D <= 512)
POWER_MAX = 0.01       # largest fraction of random-data rows with a second code inside the window (measured 2.2e-3)
RCH, KCH = 8192, 8192  # fp64 chunk: rows x codes

TC_PATHS = ("tc_small", "tc_warp")


def report(capsys, name, path, worst, amb=None, what="window ratio"):
    with capsys.disabled():
        extra = "" if amb is None else f", ambiguous rows {amb:.2e}"
        print(f"\n  [{name}] path {path}: worst {what} {worst:.3e}{extra}")


def gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def rq_path(n_select, D, ks, aligned=True, cb_aligned=True, want_train=False, tc_mode=1):
    """The kernel rq_quantize_select (csrc/rq_fused.cu) runs, for codes wanted and ks = the codebook sizes of the levels
    run.  aligned: z (and x_q / resid) 16-byte aligned; cb_aligned: every codebook run 16-byte aligned.  On the tensor
    cores, "tc_small" is the thread-per-row prepare of level 0 (D in {16, 32, 64}, aligned input), "tc_warp" the
    warp-per-row one."""
    small = D in (16, 32, 64)
    tc_ok = tc_mode != 0 and n_select >= 1024 and len(ks) > 0 and all(k >= 256 and k % 256 == 0 for k in ks) \
        and D >= 8 and D % 8 == 0
    tc = "tc_small" if small and aligned else "tc_warp"
    if tc_ok and tc_mode == 2:
        return tc
    if tc_ok and n_select >= 4096 and small and aligned and cb_aligned:
        return tc
    staged = sum(4 * (k * D + ((k + 3) & ~3)) for k in ks)
    if staged <= 200 * 1024 and aligned and cb_aligned and len(ks) > 0 and small:
        if want_train:
            return "smem_train"
        if D <= 32 and n_select >= 4096:
            return "smem_ipt4" if n_select >= 65536 else "smem_ipt2"
        return "smem_ipt1"
    if tc_ok and (any(k >= 4096 for k in ks) or D >= 128):
        return tc
    return "generic"


class pinned:
    """ops.rq_set_tc_mode(mode) inside the block, the default mode 1 afterwards"""
    def __init__(self, mode):
        self.mode = mode

    def __enter__(self):
        ops.rq_set_tc_mode(self.mode)

    def __exit__(self, *exc):
        ops.rq_set_tc_mode(1)


def misaligned(t):
    """a contiguous copy of t that starts 4 bytes into a larger buffer (a legal, non-16-byte-aligned input)"""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    assert v.data_ptr() % 16 != 0 and v.is_contiguous()
    return v


# ------------------------------------------------------------------ inputs
def make_codebooks(ks, D, seed, hostile=False):
    """randn codebooks at 0.6^l per level; hostile: code 0 zero, every 5th code (from 1) 2^-20 and (from 2) 2^20 times
    the others"""
    g = gen(seed)
    cbs = []
    for l, k in enumerate(ks):
        c = torch.randn(k, D, device=DEV, generator=g) * 0.6 ** l
        if hostile and k >= 3:
            c[0] = 0
            c[1::5] *= 2.0 ** -20
            c[2::5] *= 2.0 ** 20
        cbs.append(c)
    return cbs


def make_latents(n, D, seed, hostile=False):
    """randn rows; hostile: every 7th row zero, the others with |z| swept over 2^-56 .. 2^56 (|r|^2 finite and normal)"""
    g = gen(seed)
    z = torch.randn(n, D, device=DEV, generator=g)
    if hostile:
        e = torch.randint(-56, 57, (n, 1), device=DEV, generator=g).float()
        z = z / z.norm(dim=1, keepdim=True) * torch.exp2(e)
        z[::7] = 0
    return z


# ------------------------------------------------------------------ fp32 replay and the fp64 window
def replay(z, cbs, codes):
    """the reference's level chain in fp32 on the kernel's codes -> (residual entering each level + the last one,
    x_q, [t per level])"""
    r = z.clone()
    rs, ts, xq = [r], [], None
    for l in range(codes.shape[1]):
        q = cbs[l][codes[:, l]]
        t = q - r
        x_res = r + t
        r = r - x_res
        xq = x_res if xq is None else xq + x_res
        rs.append(r)
        ts.append(t)
    return rs, (torch.zeros_like(z) if xq is None else xq), ts


def group_max(a, group=256):
    """max |a| over each element's `group`-column scale group, zero where a is zero (exact zeros split exactly), fp64"""
    a64 = a.abs().double()
    rows, k = a64.shape
    pad = (-k) % group
    g = torch.nn.functional.pad(a64, (0, pad)).view(rows, -1, group).amax(2, keepdim=True)
    return g.expand(-1, -1, group).reshape(rows, -1)[:, :k] * (a != 0)


def window(r, cb, pick, tc):
    """-> (per-row worst ratio max_k (d64[pick] - d64[k]) / (B[k] + B[pick]), per-row 'another code in the window')"""
    n, D = r.shape
    K = cb.shape[0]
    r64, c64 = r.double(), cb.double()
    rn2, cn2 = (r64 * r64).sum(1), (c64 * c64).sum(1)
    rn, cn = rn2.sqrt(), cn2.sqrt()
    c_rel = C_TC if tc else C_SIMT * (D + 3) * U
    if tc:
        gr, r1, gc = group_max(r), r64.abs().sum(1), c64.abs().amax(1)
    cp = c64[pick]
    d_pick = rn2 + cn2[pick] - 2.0 * (r64 * cp).sum(1)
    b_pick = c_rel * (rn + cn[pick]) ** 2 + TINY
    if tc:
        b_pick = b_pick + FLOOR * ((gr * cp.abs()).sum(1) + r1 * gc[pick])
    worst = torch.full((n,), -math.inf, dtype=torch.float64, device=DEV)
    amb = torch.zeros(n, dtype=torch.bool, device=DEV)
    for i0 in range(0, n, RCH):
        i1 = min(n, i0 + RCH)
        for k0 in range(0, K, KCH):
            k1 = min(K, k0 + KCH)
            cc = c64[k0:k1]
            d = rn2[i0:i1, None] + cn2[None, k0:k1] - 2.0 * (r64[i0:i1] @ cc.t())
            b = c_rel * (rn[i0:i1, None] + cn[None, k0:k1]) ** 2 + TINY
            if tc:
                b = b + FLOOR * (gr[i0:i1] @ cc.abs().t() + r1[i0:i1, None] * gc[None, k0:k1])
            num = d_pick[i0:i1, None] - d
            den = b + b_pick[i0:i1, None]
            worst[i0:i1] = torch.maximum(worst[i0:i1], (num / den).amax(1))
            inside = num.abs() <= den
            p = pick[i0:i1]
            own = (p >= k0) & (p < k1)
            rows = torch.nonzero(own).flatten()
            inside[rows, p[rows] - k0] = False
            amb[i0:i1] |= inside.any(1)
            del d, b, num, den, inside
    return worst, amb


def check_rq(z, cbs, out, path, resid_level=-1, what=""):
    """every per-row check of the module docstring on one ops.rq_quantize result -> (worst ratio, ambiguous fraction)"""
    codes = out["codes"]
    n, run = codes.shape
    assert codes.min().item() >= 0 if n else True
    rs, xq, ts = replay(z, cbs, codes)
    if out["resid"] is not None:
        assert torch.equal(out["resid"], rs[min(resid_level, run)]), f"{what}: resid is not the replay's"
    if out["xq"] is not None:
        assert torch.equal(out["xq"], xq), f"{what}: x_q is not the replay's"
    if out["sq_err"] is not None:
        for l, t in enumerate(ts):
            want = (t * t).double().sum().item()
            got = out["sq_err"][l].item()
            assert abs(got - want) <= 1e-12 * abs(want), f"{what}: sq_err[{l}] {got!r} vs {want!r}"
    worst, amb = -math.inf, torch.zeros(n, dtype=torch.bool, device=DEV)
    for l in range(run):
        assert codes[:, l].max().item() < cbs[l].shape[0]
        w, a = window(rs[l], cbs[l], codes[:, l], path in TC_PATHS)
        if (w > 1).any():
            i = int(torch.argmax(w))
            raise AssertionError(f"{what} level {l}: {int((w > 1).sum())} rows pick outside the fp64 window, worst row {i} "
                                 f"(pick {int(codes[i, l])}, ratio {w[i].item():.3e})")
        worst = max(worst, w.max().item())
        amb |= a
    return worst, (amb.float().mean().item() if n else 0.0)


def quantize(z, cbs, mode, **kw):
    with pinned(mode):
        return ops.rq_quantize(z, cbs, **kw)


# ------------------------------------------------------------------ 1-2. path map, per-row fp64 window, exact replay
# id, n, D, ks, tc_mode, want x_q + sq_err, data, z aligned, codebooks aligned, n_levels_run (None = all), resid_level,
# the path the case is for
CASES = [
    ("ipt1_n1", 1, 32, [256] * 4, 1, False, "randn", True, True, None, 0, "smem_ipt1"),
    ("ipt1_n255_hostile", 255, 32, [256] * 4, 1, False, "hostile", True, True, None, 4, "smem_ipt1"),
    ("ipt1_n256_mixed_k", 256, 16, [256, 200, 3, 1], 0, False, "randn", True, True, None, 2, "smem_ipt1"),
    ("ipt1_n257_d64", 257, 64, [256] * 2, 1, False, "randn", True, True, None, 1, "smem_ipt1"),
    ("ipt1_n1023_run1", 1023, 32, [512, 256], 1, False, "randn", True, True, 1, 1, "smem_ipt1"),
    ("ipt1_d64_n70001", 70001, 64, [200] * 2, 1, False, "randn", True, True, None, 2, "smem_ipt1"),
    ("train_n1024", 1024, 32, [256] * 4, 1, True, "randn", True, True, None, 3, "smem_train"),
    ("train_n4095_d64_hostile", 4095, 64, [256, 256], 1, True, "hostile", True, True, None, 2, "smem_train"),
    ("ipt2_n4096_d16", 4096, 16, [256] * 4, 0, False, "randn", True, True, None, 4, "smem_ipt2"),
    ("ipt2_l8_run6", 4096, 16, [256, 3, 200, 1, 256, 512, 5, 64], 1, False, "randn", True, True, 6, 3, "smem_ipt2"),
    ("ipt2_n65535", 65535, 32, [256] * 4, 0, False, "randn", True, True, None, 4, "smem_ipt2"),
    ("ipt4_n65536", 65536, 32, [256] * 4, 0, False, "randn", True, True, None, 4, "smem_ipt4"),
    ("ipt4_n70001_k200", 70001, 16, [200] * 3, 1, False, "hostile", True, True, None, 3, "smem_ipt4"),
    ("generic_d5", 1023, 5, [3, 1, 200], 1, True, "hostile", True, True, None, 3, "generic"),
    ("generic_d24_k1", 4096, 24, [1, 256, 1], 1, True, "randn", True, True, None, 2, "generic"),
    ("generic_d24", 4096, 24, [256] * 4, 0, False, "randn", True, True, None, 4, "generic"),
    ("generic_d40", 1024, 40, [512, 256], 0, False, "randn", True, True, None, 1, "generic"),
    ("generic_d128", 4097, 128, [256] * 4, 0, True, "randn", True, True, None, 4, "generic"),
    ("generic_staged_1mb", 1024, 64, [1024] * 4, 0, False, "randn", True, True, None, 4, "generic"),
    ("generic_k8192_n257", 257, 256, [8192, 256], 1, False, "randn", True, True, None, 2, "generic"),
    ("generic_misaligned_z", 4096, 32, [256] * 4, 1, True, "randn", False, True, None, 4, "generic"),
    ("generic_misaligned_cb", 70001, 16, [256] * 2, 1, False, "randn", True, False, None, 2, "generic"),
    ("tc_small_n4096", 4096, 32, [256] * 4, 1, False, "randn", True, True, None, 4, "tc_small"),
    ("tc_small_train", 4096, 32, [256] * 4, 1, True, "hostile", True, True, None, 2, "tc_small"),
    ("tc_small_d64_n65536", 65536, 64, [512, 256], 1, False, "randn", True, True, None, 1, "tc_small"),
    ("tc_small_l8_n70001", 70001, 16, [256, 512, 256, 1024, 256, 256, 768, 256], 1, True, "randn", True, True, None, 8,
     "tc_small"),
    ("tc_small_k4096_n1024", 1024, 32, [4096, 256], 1, False, "randn", True, True, None, 2, "tc_small"),
    ("tc_d8", 1024, 8, [256, 256], 2, True, "randn", True, True, None, 1, "tc_warp"),
    ("tc_d24_n4095", 4095, 24, [256] * 3, 2, True, "hostile", True, True, None, 3, "tc_warp"),
    ("tc_d40", 2000, 40, [512, 256], 2, False, "randn", True, True, None, 2, "tc_warp"),
    ("tc_d128", 4096, 128, [256] * 4, 1, False, "randn", True, True, 3, 2, "tc_warp"),
    ("tc_d256_k4096", 4096, 256, [4096, 4096], 1, False, "randn", True, True, None, 2, "tc_warp"),
    ("tc_d264_hostile", 1024, 264, [256, 512], 1, True, "hostile", True, True, None, 1, "tc_warp"),
    ("tc_d264", 4097, 264, [256, 512], 1, False, "randn", True, True, None, 2, "tc_warp"),
    ("tc_d512", 4097, 512, [256, 256], 1, True, "randn", True, True, None, 2, "tc_warp"),
    ("tc_k8192_n1024", 1024, 256, [8192], 1, False, "randn", True, True, None, 0, "tc_warp"),
    ("tc_misaligned_z_d256", 1024, 256, [256, 256], 1, False, "randn", False, True, None, 2, "tc_warp"),
    ("tc_misaligned_z_k4096", 1024, 32, [4096, 256], 1, True, "randn", False, True, None, 1, "tc_warp"),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_rq_rows_against_fp64(case, capsys):
    name, n, D, ks, mode, train, kind, z_al, cb_al, run, resid_level, path = case
    run_ks = ks if run is None else ks[:run]
    assert rq_path(n, D, run_ks, z_al, cb_al, train, mode) == path
    hostile = kind == "hostile"
    cbs = make_codebooks(ks, D, seed=n + D + len(ks), hostile=hostile)
    z = make_latents(n, D, seed=n * 7 + D, hostile=hostile)
    zi = z if z_al else misaligned(z)
    cbi = cbs if cb_al else [misaligned(c) for c in cbs]
    out = quantize(zi, cbi, mode, n_levels_run=run, resid_level=resid_level, want_xq=train, want_sq_err=train)
    assert out["codes"].shape == (n, len(run_ks))
    worst, amb = check_rq(z, cbs, out, path, resid_level, name)
    report(capsys, name, path, worst, amb)
    if kind == "randn" and n >= 1000:
        assert amb < POWER_MAX, f"{name}: {amb:.3%} of the rows hold a second code inside the window"


# ------------------------------------------------------------------ exact ties
DUP0 = [(5, 200), (130, 131), (100, 300), (10, 460), (255, 256)]     # K = 512: across column halves, tiles, neighbours
DUP1 = [(0, 255), (3, 128), (64, 65)]
TIE_CASES = [  # id, n, D, tc_mode, want_xq, path
    ("smem_ipt1", 1000, 32, 0, False, "smem_ipt1"),
    ("smem_ipt2", 5000, 32, 0, False, "smem_ipt2"),
    ("smem_ipt4", 70001, 32, 0, False, "smem_ipt4"),
    ("smem_train", 5000, 32, 0, True, "smem_train"),
    ("generic", 5000, 24, 0, True, "generic"),
    ("tc_small", 5000, 32, 1, True, "tc_small"),
    ("tc_warp_d24", 5000, 24, 2, True, "tc_warp"),
    ("tc_warp_d264", 5000, 264, 1, False, "tc_warp"),
]


@pytest.mark.parametrize("case", TIE_CASES, ids=[c[0] for c in TIE_CASES])
def test_exact_ties_keep_the_lower_index(case, capsys):
    """codebooks with duplicated code rows and a batch with duplicated rows: the higher copy of a duplicate code is
    never picked, and duplicate rows get identical codes, residuals and x_q"""
    name, n, D, mode, train, path = case
    ks = [512, 256]
    assert rq_path(n, D, ks, want_train=train, tc_mode=mode) == path
    g = gen(97)
    cbs = [torch.randn(512, D, device=DEV, generator=g), torch.randn(256, D, device=DEV, generator=g) * 1e-3]
    for cb, dups in ((cbs[0], DUP0), (cbs[1], DUP1)):
        for i, j in dups:
            cb[j] = cb[i]
    lo0 = torch.tensor([i for i, _ in DUP0], device=DEV)
    lo1 = torch.tensor([i for i, _ in DUP1], device=DEV)
    a = lo0[torch.randint(0, len(DUP0), (n,), device=DEV, generator=g)]
    b = lo1[torch.randint(0, len(DUP1), (n,), device=DEV, generator=g)]
    z = cbs[0][a] + cbs[1][b] + 1e-5 * torch.randn(n, D, device=DEV, generator=g)
    half = n // 2
    z[half:] = torch.randn(n - half, D, device=DEV, generator=g)                     # and rows that pick anything
    p = torch.randperm(n, device=DEV, generator=g)
    p = p[(p != 0) & (p != 1) & (p != 256) & (p != n - 1)]
    src, dst = p[: n // 10], p[n // 10: n // 5]                                      # disjoint: each copy has one source
    z[dst] = z[src]
    z[-1] = z[0]
    z[256] = z[1]
    out = quantize(z, cbs, mode, resid_level=2, want_xq=train)
    codes = out["codes"]
    for l, dups in enumerate((DUP0, DUP1)):
        for i, j in dups:
            assert not (codes[:, l] == j).any(), f"{name}: level {l} picks the higher copy {j} of code {i}"
        assert torch.isin(codes[:, l], torch.tensor([i for i, _ in dups], device=DEV)).float().mean() > 0.3
    for k in (codes, out["resid"]) + ((out["xq"],) if train else ()):
        assert torch.equal(k[dst], k[src]) and torch.equal(k[-1], k[0]) and torch.equal(k[256], k[1])
    worst, _ = check_rq(z, cbs, out, path, 2, name)
    report(capsys, f"ties {name}", path, worst)


# ------------------------------------------------------------------ 3. bit-exact invariances
@pytest.mark.parametrize("D,ks", [(32, [256] * 4), (16, [200] * 3)])
def test_smem_family_rows_are_identical(D, ks):
    """the same row from IPT 4 (70 001 rows), IPT 2 (5 000), IPT 1 (1 000) and TRAIN (x_q wanted): identical codes and
    residuals, which pins each kernel's item-to-thread mapping"""
    n = 70001
    cbs = make_codebooks(ks, D, seed=3)
    z = make_latents(n, D, seed=4)
    L = len(ks)
    with pinned(0):
        assert rq_path(n, D, ks, tc_mode=0) == "smem_ipt4"
        full = ops.rq_quantize(z, cbs, resid_level=L)
        assert rq_path(n, D, ks, want_train=True, tc_mode=0) == "smem_train"
        train = ops.rq_quantize(z, cbs, resid_level=L, want_xq=True)
        assert torch.equal(train["codes"], full["codes"]) and torch.equal(train["resid"], full["resid"])
        p = torch.randperm(n, device=DEV, generator=gen(5))
        for m, path in ((5000, "smem_ipt2"), (1000, "smem_ipt1")):
            assert rq_path(m, D, ks, tc_mode=0) == path
            idx = p[:m]
            sub = ops.rq_quantize(z[idx], cbs, resid_level=L)
            assert torch.equal(sub["codes"], full["codes"][idx]), path
            assert torch.equal(sub["resid"], full["resid"][idx]), path
    rs, _, _ = replay(z, cbs, full["codes"])
    assert torch.equal(full["resid"], rs[L])


@pytest.mark.parametrize("D,ks", [(32, [256] * 4), (264, [256, 512])])
def test_tensor_core_rows_are_independent(D, ks):
    """tc_mode 2: a row permutation and subsets of >= 1024 rows give bit-identical codes and residuals"""
    n = 5000
    cbs = make_codebooks(ks, D, seed=6)
    z = make_latents(n, D, seed=7)
    L = len(ks)
    with pinned(2):
        full = ops.rq_quantize(z, cbs, resid_level=L)
        p = torch.randperm(n, device=DEV, generator=gen(8))
        perm = ops.rq_quantize(z[p], cbs, resid_level=L)
        assert torch.equal(perm["codes"], full["codes"][p]) and torch.equal(perm["resid"], full["resid"][p])
        for a, b in ((0, 1024), (1000, 2100), (3976, 5000)):
            assert rq_path(b - a, D, ks, tc_mode=2) in TC_PATHS
            sub = ops.rq_quantize(z[a:b], cbs, resid_level=L)
            assert torch.equal(sub["codes"], full["codes"][a:b]) and torch.equal(sub["resid"], full["resid"][a:b]), (a, b)
        idx = p[:1024]
        sub = ops.rq_quantize(z[idx], cbs, resid_level=L)
        assert torch.equal(sub["codes"], full["codes"][idx]) and torch.equal(sub["resid"], full["resid"][idx])


SCALE_CASES = [  # n, D, ks, tc_mode, want_xq, path
    (65536, 16, [200] * 3, 0, False, "smem_ipt4"),
    (5000, 32, [256] * 4, 0, False, "smem_ipt2"),
    (1000, 32, [256] * 4, 0, False, "smem_ipt1"),
    (1000, 32, [256] * 4, 0, True, "smem_train"),
    (1500, 24, [256, 3], 1, True, "generic"),
    (4096, 32, [256] * 4, 1, True, "tc_small"),
    (1024, 264, [256, 512], 1, True, "tc_warp"),
    (2048, 8, [256, 256], 2, False, "tc_warp"),
]


@pytest.mark.parametrize("case", SCALE_CASES, ids=[c[-1] + f"_d{c[1]}" for c in SCALE_CASES])
def test_power_of_two_scaling_is_exact(case):
    """z and codebooks times 2^s: identical codes, residuals and x_q times 2^s, bit for bit.  s keeps |r|^2, |c_k|^2
    and every non-zero product r_d c_kd normal (randn entries >= 2^-27, products scale by 2^2s), far from the +-126
    clamp of the tensor-core split scales"""
    n, D, ks, mode, train, path = case
    assert rq_path(n, D, ks, want_train=train, tc_mode=mode) == path
    cbs = make_codebooks(ks, D, seed=9)
    z = make_latents(n, D, seed=10)
    L = len(ks)
    base = quantize(z, cbs, mode, resid_level=L, want_xq=train)
    for s in (-30, -7, 11, 40):
        f = 2.0 ** s
        out = quantize(z * f, [c * f for c in cbs], mode, resid_level=L, want_xq=train)
        assert torch.equal(out["codes"], base["codes"]), s
        assert torch.equal(out["resid"], base["resid"] * f), s
        if train:
            assert torch.equal(out["xq"], base["xq"] * f), s


def test_near_tie_disagreement_is_inside_both_windows(capsys):
    """latents at the midpoints of pairs of level-0 codes, pushed off the tie by 1e-8 .. 1e-4: the SIMT and tensor-core
    paths pick differently on some rows, and each pick is inside its own path's fp64 window on every row"""
    n, D, ks = 20000, 32, [256] * 4
    cbs = make_codebooks(ks, D, seed=11)
    g = gen(12)
    a = torch.randint(0, ks[0], (n,), device=DEV, generator=g)
    b = torch.randint(0, ks[0], (n,), device=DEV, generator=g)
    noise = 10.0 ** (-8 + 4 * torch.rand((n, 1), device=DEV, generator=g))
    z = (cbs[0][a] + cbs[0][b]) / 2 + noise * torch.randn(n, D, device=DEV, generator=g)
    assert rq_path(n, D, ks, tc_mode=0) == "smem_ipt2" and rq_path(n, D, ks, tc_mode=2) == "tc_small"
    simt = quantize(z, cbs, 0, resid_level=len(ks))
    tc = quantize(z, cbs, 2, resid_level=len(ks))
    differ = int((simt["codes"] != tc["codes"]).any(1).sum())
    w_simt, _ = check_rq(z, cbs, simt, "smem_ipt2", len(ks), "near-tie SIMT")
    w_tc, _ = check_rq(z, cbs, tc, "tc_small", len(ks), "near-tie TC")
    with capsys.disabled():
        print(f"\n  [near-tie] {differ} of {n} rows differ between SIMT and tensor-core codes")
    report(capsys, "near-tie SIMT", "smem_ipt2", w_simt)
    report(capsys, "near-tie TC", "tc_small", w_tc)
    assert differ > 0, "no near-tie separates the SIMT and tensor-core paths"


# ------------------------------------------------------------------ vq_distances
@pytest.mark.parametrize("n,D,K,hostile", [(1, 5, 1, False), (257, 33, 300, False), (1000, 256, 512, False),
                                           (64, 512, 8192, False), (700, 32, 256, True)])
def test_vq_distances_per_element(n, D, K, hostile, capsys):
    """every distance of vq_distances_kernel against fp64 with the SIMT bound B[k]"""
    r = make_latents(n, D, seed=n + D, hostile=hostile)
    cb = make_codebooks([K], D, seed=K + D, hostile=hostile)[0]
    d = ops.vq_distances(r, cb)
    r64, c64 = r.double(), cb.double()
    rn2, cn2 = (r64 * r64).sum(1), (c64 * c64).sum(1)
    d64 = rn2[:, None] + cn2[None, :] - 2.0 * (r64 @ c64.t())
    bnd = C_SIMT * (D + 3) * U * (rn2.sqrt()[:, None] + cn2.sqrt()[None, :]) ** 2 + TINY
    err = (d.double() - d64).abs()
    bad = ~(err <= bnd)
    assert not bad.any(), f"{int(bad.sum())} distances over the bound, first {bad.nonzero()[0].tolist()}"
    report(capsys, f"vq_distances n={n} D={D} K={K} hostile={hostile}", "vq_distances", (err / bnd).max().item(),
           what="|d - d64| / B")


# ------------------------------------------------------------------ 5. training forward / backward
def ulp32(x64):
    """fp32 unit in the last place at the fp64 values x64"""
    e = torch.frexp(x64.abs()).exponent
    return torch.where(x64 == 0, 2.0 ** -149, torch.exp2((e - 24).clamp(min=-149).double()))


def check_train(z, codes, cbs, g_xq, g_loss, beta0, capsys, what):
    """rq_train_forward / rq_train_backward against their sequential fp32 replays and fp64"""
    n, D = z.shape
    L = len(cbs)
    ks = [c.shape[0] for c in cbs]
    fw = ops.rq_train_forward(z, codes, cbs)
    rs, xq, ts = replay(z, cbs, codes)
    assert torch.equal(fw["xq"], xq), f"{what}: x_q"
    for l in range(L):
        assert torch.equal(fw["diffs"][l], ts[l]), f"{what}: diffs[{l}]"
        want = (ts[l].double() ** 2).sum().item()
        assert abs(fw["sq_err"][l].item() - want) <= 1e-12 * want, f"{what}: sq_err[{l}]"
    assert torch.equal(fw["codes_t"], codes.t())

    gz, gcb = ops.rq_train_backward(fw["diffs"], fw["codes_t"], ks, g_xq, g_loss, beta0)
    per_elem = 2.0 / (float(n) * float(D)) / L
    gl = np.float32(g_loss.item())
    scale = np.float32(gl * np.float32(per_elem))
    diffs = fw["diffs"].cpu().numpy()
    cdx = codes.cpu().numpy()
    worst = 0.0
    for l in range(L):
        acc = np.zeros((ks[l], D), dtype=np.float32)
        np.add.at(acc, cdx[:, l], diffs[l])                       # unbuffered: fp32 adds in item order
        want = acc * scale
        got = gcb[l].cpu().numpy()
        assert np.array_equal(got, want), f"{what}: codebook gradient {l} differs from the item-order fp32 sum"
        s64 = np.zeros((ks[l], D))
        a64 = np.zeros((ks[l], D))
        np.add.at(s64, cdx[:, l], diffs[l].astype(np.float64))
        np.add.at(a64, cdx[:, l], np.abs(diffs[l]).astype(np.float64))
        cnt = np.bincount(cdx[:, l], minlength=ks[l]).astype(np.float64)[:, None]
        g64 = s64 * float(scale)
        bnd = abs(float(scale)) * cnt * U * a64 + U * np.abs(g64) + 2.0 ** -149
        err = np.abs(got.astype(np.float64) - g64)
        assert (err <= bnd).all(), f"{what}: codebook gradient {l} off the fp64 sum"
        worst = max(worst, float((err / bnd).max()))
        assert (got[cnt[:, 0] == 0] == 0).all()
    scale_z = np.float32(gl * np.float32(-beta0 * per_elem))
    v64 = fw["diffs"][0].double() * float(scale_z) + (0.0 if g_xq is None else g_xq.double())
    assert ((gz.double() - v64).abs() <= ulp32(v64)).all(), f"{what}: g_z more than 1 ulp off fp64"
    # no loss gradient: exact zeros and g_z == g_xq
    gz0, gcb0 = ops.rq_train_backward(fw["diffs"], fw["codes_t"], ks, g_xq, None, beta0)
    assert all((g == 0).all() for g in gcb0)
    assert torch.equal(gz0, torch.zeros_like(gz0) if g_xq is None else g_xq)
    report(capsys, what, "rq_train", worst, what="codebook gradient |g - g64| / (count 2^-24 sum |diff|)")


def random_codes(n, ks, seed, empty_every=0):
    g = gen(seed)
    cols = []
    for k in ks:
        c = torch.randint(0, k, (n,), device=DEV, generator=g)
        if empty_every and k > empty_every:
            c = torch.where(c % empty_every == 0, (c + 1) % k, c)          # codes k % empty_every == 0 stay empty
        cols.append(c)
    return torch.stack(cols, 1)


@pytest.mark.parametrize("members", [1919, 1920, 1921, 2048, 5000])
def test_train_one_code_with_many_members(members, capsys):
    """one code of level 0 holding `members` consecutive rows and one of level 1 holding as many scattered rows: the
    ordered sum's flush (kSegList - kSegThreads = 1920 buffered members) at, below and above its threshold and several
    times over; codes without members; member counts of every residue mod 4 (the flush's scalar tail)"""
    n, D, ks = members + 1237, 33, [16, 300]
    g = gen(members)
    codes = random_codes(n, ks, seed=members + 1, empty_every=4)
    codes[:, 0] = torch.where(codes[:, 0] == 5, 6, codes[:, 0])
    start = 301
    codes[start:start + members, 0] = 5
    codes[:, 1] = torch.where(codes[:, 1] == 7, 9, codes[:, 1])
    codes[torch.randperm(n, device=DEV, generator=g)[:members], 1] = 7
    counts = [torch.bincount(codes[:, l], minlength=k) for l, k in enumerate(ks)]
    assert int(counts[0][5]) == members and int(counts[1][7]) == members
    res = set(int(x) % 4 for x in counts[1][counts[1] > 0].tolist())
    assert {1, 2, 3} <= res and (counts[1] == 0).any()
    cbs = make_codebooks(ks, D, seed=members + 2)
    z = make_latents(n, D, seed=members + 3)
    g_xq = torch.randn(n, D, device=DEV, generator=g)
    check_train(z, codes, cbs, g_xq, torch.tensor(0.7312, device=DEV), 0.25, capsys, f"train members={members}")


@pytest.mark.parametrize("n,D,ks,with_gxq", [
    (1, 1, [4], True),
    (999, 1, [256, 3, 200, 1, 512, 5, 64, 1024], True),
    (1000, 33, [256, 3, 200, 1, 512, 5, 64, 1024], False),
    (1003, 33, [300], True),
    (2049, 8192, [7, 300], True),
    (130, 8192, [2, 5, 3, 1, 4, 6, 8, 7], False),
])
def test_train_forward_backward_exact(n, D, ks, with_gxq, capsys):
    """L = 1 and 8 with mixed K (the first_block level lookup), e_dim 1 / 33 / 8192 (the backward's limit), n not a
    multiple of 8 or 128, no g_xq"""
    cbs = make_codebooks(ks, D, seed=n + D)
    z = make_latents(n, D, seed=n + D + 1)
    codes = random_codes(n, ks, seed=n + D + 2, empty_every=3)
    g_xq = torch.randn(n, D, device=DEV, generator=gen(n)) if with_gxq else None
    check_train(z, codes, cbs, g_xq, torch.tensor(-1.37, device=DEV), 0.25, capsys, f"train n={n} D={D} L={len(ks)}")
