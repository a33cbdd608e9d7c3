"""Index generation over the GPUs of a box from the generate_indices CLI (B200): the JSON fragments of row blocks
(lcrec_index_json_ex), PASS 0 of a host block in the pieces of the one-GPU run (lcrec_indexer_pass0_host_ex), and the CLI
under torchrun against the one-GPU CLI, byte for byte - including a checkpoint whose bucket skew overflows the native
exchange's slabs, which every rank then leaves together for the split-size path."""
import argparse
import contextlib
import io
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from lcrec_b200.distributed import ShardPlan, bucket_owner
from lcrec_b200.synth import seeded_weights, synth_items

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from lcrec_b200 import ops
    from lcrec_b200 import generate_indices as G
    from lcrec_b200.models import RQVAE
    DEV = torch.device("cuda:0")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_GPUS = torch.cuda.device_count() if torch.cuda.is_available() else 0
multi_gpu = pytest.mark.skipif(N_GPUS < 2, reason="needs 2 GPUs")


def _dump(codes, base=0):
    return json.dumps({base + i: [G.PREFIX[l].format(int(v)) for l, v in enumerate(row)] for i, row in enumerate(codes.tolist())})


# ------------------------------------------------------------------ 1. JSON fragments
@pytest.mark.parametrize("n,L,cuts", [
    (0, 3, [0, 0]), (1, 4, [0, 0, 1, 1]), (25, 1, [0, 9, 10, 25]), (250, 2, [0, 99, 100, 100, 250]),
    (100005, 5, [0, 9, 10, 99, 100, 99999, 100000, 100005]), (4097, 4, [0, 1024, 3000, 4097]), (777, 3, [0, 777])])
def test_fragments_concatenate_to_the_table(n, L, cuts):
    rng = np.random.default_rng(n + 7 * L)
    codes = rng.integers(0, 8192, size=(n, L)).astype(np.int64)
    if n > 3:
        codes[1] = 0; codes[2] = 8191
    cd = torch.from_numpy(codes).to(DEV)
    whole = ops.index_json_bytes(cd)
    assert whole == _dump(codes).encode()
    body = b"".join(ops.index_json_bytes(cd[a:b], item_base=a, braces=False) for a, b in zip(cuts[:-1], cuts[1:]))
    assert b"{" + body + b"}" == whole
    assert ops.index_json_bytes(cd[:0], item_base=5, braces=False) == b""


@pytest.mark.parametrize("L", [1, 2, 3, 4, 5])
def test_fragment_keys_past_2_31(L):
    base = (1 << 31) + 5                                            # int64 keys: the digit counts hold past 2^31
    codes = np.random.default_rng(L).integers(0, 256, size=(1500, L)).astype(np.int64)
    got = ops.index_json_bytes(torch.from_numpy(codes).to(DEV), item_base=base, braces=False)
    assert got == (", " + _dump(codes, base)[1:-1]).encode()
    got = ops.index_json_bytes(torch.from_numpy(codes).to(DEV), item_base=base - 1000, braces=True)
    assert got == b"{" + (", " + _dump(codes, base - 1000)[1:-1]).encode() + b"}"      # key != 0: ", " before it, braces or not


# ------------------------------------------------------------------ 2. piece-aligned PASS 0
IN_DIM, E_DIM, K = 32, 32, 256


def _tie_model():
    """Encoder = identity (relu(x) - relu(-x) through a 64-wide hidden layer; the weights are exact in every split), four
    256 x 32 codebooks of small dyadic values, so a latent can sit at (nearly) the midpoint of two level-0 codes."""
    m = RQVAE(in_dim=IN_DIM, num_emb_list=[K] * 4, e_dim=E_DIM, layers=[2 * IN_DIM], sk_epsilons=[0.0, 0.0, 0.0, 0.003], sk_iters=50)
    sd = m.state_dict()
    eye = torch.eye(IN_DIM)
    sd["encoder.mlp_layers.1.weight"] = torch.cat([eye, -eye], 0)
    sd["encoder.mlp_layers.1.bias"] = torch.zeros(2 * IN_DIM)
    sd["encoder.mlp_layers.4.weight"] = torch.cat([eye, -eye], 1)
    sd["encoder.mlp_layers.4.bias"] = torch.zeros(IN_DIM)
    g = torch.Generator().manual_seed(4)
    cbs = []
    for l in range(4):
        cb = torch.randint(-64, 65, (K, E_DIM), generator=g).float() / (64.0 * 2 ** l)
        sd[f"rq.vq_layers.{l}.embedding.weight"] = cb
        cbs.append(cb)
    m.load_state_dict(sd)
    return m.to(DEV).eval(), cbs


def _tie_items(n, cb0, seed):
    """Latents at the midpoints of random pairs of level-0 codes, pushed off the tie by noise of 1e-8 .. 1e-4."""
    g = torch.Generator().manual_seed(seed)
    a, b = torch.randint(0, K, (n,), generator=g), torch.randint(0, K, (n,), generator=g)
    mid = (cb0[a] + cb0[b]) / 2
    scale = 10.0 ** (-8 + 4 * torch.rand((n, 1), generator=g))
    return (mid + scale * torch.randn((n, E_DIM), generator=g)).numpy().astype(np.float32)


@pytest.fixture(scope="module")
def tie_setup():
    m, cbs = _tie_model()
    x = _tie_items(23001, cbs[0], 1)
    # the two RQ paths really disagree on some of these rows: otherwise the test below could not see the layout
    with torch.no_grad():
        z = m.encoder._get_handle().forward(torch.from_numpy(x).to(DEV))
    cbd = [c.to(DEV) for c in cbs]
    try:
        ops.rq_set_tc_mode(0)
        simt = ops.rq_quantize(z, cbd)["codes"]
        ops.rq_set_tc_mode(2)
        tc = ops.rq_quantize(z, cbd)["codes"]
    finally:
        ops.rq_set_tc_mode(1)
    n_disagree = int((simt != tc).any(dim=1).sum())
    assert n_disagree > 0, "no near-tie separates the SIMT and tensor-core RQ paths"
    return m, x, n_disagree


def _host_input(x32, dtype, kind, tmp_path):
    if dtype == torch.bfloat16:
        t = torch.from_numpy(x32).to(torch.bfloat16)
        return t.pin_memory() if kind == "pinned" else t
    arr = x32.astype(np.float16 if dtype == torch.float16 else np.float32)
    if kind == "memmap":
        np.save(tmp_path / "x.npy", arr)
        return np.load(tmp_path / "x.npy", mmap_mode="r")
    if kind == "pinned":
        return torch.from_numpy(arr).pin_memory()
    return arr


@pytest.mark.parametrize("dtype,kind", [(torch.float32, "pageable"), (torch.float32, "memmap"), (torch.float32, "pinned"),
                                        (torch.float16, "pageable"), (torch.float16, "memmap"), (torch.float16, "pinned"),
                                        (torch.bfloat16, "pageable"), (torch.bfloat16, "pinned")])
def test_pass0_host_blocks_equal_one_gpu_table(tie_setup, dtype, kind, tmp_path):
    """Ranks 2..8 of ShardPlan blocks, chunks of 5000 rows: pieces of >= 4096 rows (tensor-core RQ path) that a block meets
    in fewer rows, and a last piece of 3001 rows (SIMT path) - every block's rows equal the one-GPU PASS-0 table."""
    m, x32, _ = tie_setup
    n, chunk = x32.shape[0], 5000
    xh = _host_input(x32, dtype, kind, tmp_path)
    ref_ix = G.build_indexer(m, n, chunk)
    ref_codes, _ = ref_ix.run_host(xh if not isinstance(xh, np.ndarray) else torch.from_numpy(np.ascontiguousarray(xh)),
                                   max_rounds=0)                      # run_host's PASS-0 table: no round rewrites it
    ref_resid = ref_ix.resid_view(n).clone()
    ix = G.build_indexer(m, n, chunk)
    without_hint = 0
    for world in range(2, 9):
        plan = ShardPlan(n, world)
        for r in range(world):
            sl = plan.slice(r)
            ix.pass0_host(xh[sl], n, plan.start(r))
            k = plan.count(r)
            assert torch.equal(ix.codes_view(k).cpu(), ref_codes[sl]), (world, r)
            assert torch.equal(ix.resid_view(k), ref_resid[sl]), (world, r)
        if dtype == torch.float32 and kind == "pageable":
            # the same cut with each part choosing its RQ path from its own row count (no hint) differs from one GPU
            xd = torch.from_numpy(x32).to(DEV)
            for r in range(world):
                s0, e0 = plan.start(r), plan.start(r) + plan.count(r)
                for p0 in range(0, n, chunk):
                    s, e = max(p0, s0), min(p0 + chunk, e0)
                    if s < e:
                        ix.pass0(xd[s:e], s - s0)
                without_hint += int((ix.codes_view(e0 - s0).cpu() != ref_codes[s0:e0]).any(dim=1).sum())
    if dtype == torch.float32 and kind == "pageable":
        assert without_hint > 0


def test_pass0_host_refuses_more_rows_than_the_table(tie_setup):
    m, x32, _ = tie_setup
    ix = G.build_indexer(m, 1000, 500)
    with pytest.raises(RuntimeError, match="invalid argument"):
        ix.pass0_host(x32[:1001], 5000, 10)


RUNSH_DIMS = [4096, 2048, 1024, 512, 256, 128, 64, 32]


@pytest.fixture(scope="module")
def runsh():
    ws, bs, cbs = seeded_weights(RUNSH_DIMS, [256] * 4, 32, seed=3, cb_scale=0.02)
    m = RQVAE(in_dim=4096, num_emb_list=[256] * 4, e_dim=32, layers=RUNSH_DIMS[1:-1], sk_epsilons=[0.0, 0.0, 0.0, 0.003], sk_iters=50)
    sd = m.state_dict()
    lin = sorted([k for k in sd if k.startswith("encoder.mlp_layers.") and k.endswith(".weight")], key=lambda s: int(s.split(".")[2]))
    for k, w, b in zip(lin, ws, bs):
        sd[k] = torch.from_numpy(w); sd[k.replace(".weight", ".bias")] = torch.from_numpy(b)
    for l, cb in enumerate(cbs):
        sd[f"rq.vq_layers.{l}.embedding.weight"] = torch.from_numpy(cb)
    m.load_state_dict(sd)
    return m.to(DEV).eval()


@pytest.mark.parametrize("n,chunk,dtype,launches", [(50000, 16384, np.float32, 764), (50000, 32768, np.float16, 754),
                                                    (3001, 1024, np.float32, 366)])
def test_run_host_launch_count(runsh, n, chunk, dtype, launches):
    """run_host = pass0_host(n, 0, n) + rounds + D2H: the kernel launches of a whole run_host call (PASS 0 and the 20
    rounds) are the counts the library made for these inputs before run_host was rebuilt on pass0_host (B200)."""
    x = torch.from_numpy(synth_items(n, 4096, n_parents=n // 8, seed=12).astype(dtype))
    ix = G.build_indexer(runsh, n, chunk)
    ix.run_host(x, max_rounds=20)                                # lazily created state (copy stream, round graphs)
    torch.cuda.synchronize()
    l0 = ops.launch_count()
    ix.run_host(x, max_rounds=20)
    torch.cuda.synchronize()
    assert ops.launch_count() - l0 == launches


def test_pass0_host_back_to_back_calls(runsh):
    """Two blocks through one indexer with no synchronisation in between: the second call's first copies must not land in
    the staging buffers while the first call's last encoder passes still read them.  Rows [8192, 40000) of the table keep
    the first block's results (the second block writes rows [0, 8192))."""
    n, chunk = 48192, 8192
    x = torch.from_numpy(synth_items(n, 4096, n_parents=n // 8, seed=31)).pin_memory()
    ref = G.build_indexer(runsh, n, chunk)
    ref.pass0_host(x[:40000], n, 0)
    torch.cuda.synchronize()
    want_a = (ref.codes_view(40000)[8192:].clone(), ref.resid_view(40000)[8192:].clone())
    ref.pass0_host(x[40000:], n, 40000)
    torch.cuda.synchronize()
    want_b = (ref.codes_view(8192).clone(), ref.resid_view(8192).clone())
    ix = G.build_indexer(runsh, n, chunk)
    for _ in range(3):
        ix.pass0_host(x[:40000], n, 0)
        ix.pass0_host(x[40000:], n, 40000)                       # no host or device synchronisation between the calls
        torch.cuda.synchronize()
        assert torch.equal(ix.codes_view(40000)[8192:], want_a[0]) and torch.equal(ix.resid_view(40000)[8192:], want_a[1])
        assert torch.equal(ix.codes_view(8192), want_b[0]) and torch.equal(ix.resid_view(8192), want_b[1])


# ------------------------------------------------------------------ 3. the CLI under torchrun
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _torchrun(*argv, nproc=2, timeout=900):
    return subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc), "--master-addr",
                           "127.0.0.1", "--master-port", str(_free_port()), *argv],
                          capture_output=True, text=True, timeout=timeout, cwd=ROOT)


def _stat_lines(text):
    return [l for l in text.splitlines() if l.startswith(("All indices number", "Max number of conflicts", "Collision Rate"))]


def _checkpoint(tmp_path, num_emb_list, dims, skew=False, seed=3):
    """A seeded checkpoint; ``skew``: level 0 can only pick codes whose bucket owner is rank 0 for 2 and 8 ranks (the other
    codes sit far away), so every item goes to one rank and the native exchange's slabs overflow."""
    ws, bs, cbs = seeded_weights(dims, num_emb_list, dims[-1], seed=seed, cb_scale=0.02)
    L = len(num_emb_list)
    m = RQVAE(in_dim=dims[0], num_emb_list=num_emb_list, e_dim=dims[-1], layers=dims[1:-1], sk_epsilons=[0.0] * (L - 1) + [0.003],
              sk_iters=50)
    sd = m.state_dict()
    lin = sorted([k for k in sd if k.startswith("encoder.mlp_layers.") and k.endswith(".weight")], key=lambda s: int(s.split(".")[2]))
    for k, w, b in zip(lin, ws, bs):
        sd[k] = torch.from_numpy(w); sd[k.replace(".weight", ".bias")] = torch.from_numpy(b)
    for l, cb in enumerate(cbs):
        cb = torch.from_numpy(cb)
        if skew and l == 0:
            codes = torch.zeros((num_emb_list[0], L), dtype=torch.int64)
            codes[:, 0] = torch.arange(num_emb_list[0])
            far = bucket_owner(codes, num_emb_list, 8) != 0
            cb[far] = 1000.0
        sd[f"rq.vq_layers.{l}.embedding.weight"] = cb
    m.load_state_dict(sd)
    args = argparse.Namespace(data_path="unused.npy", num_emb_list=num_emb_list, e_dim=dims[-1], layers=dims[1:-1], dropout_prob=0.0,
                              bn=False, loss_type="mse", quant_loss_weight=1.0, kmeans_init=False, kmeans_iters=100,
                              sk_epsilons=[0.0] * (L - 1) + [0.003], sk_iters=50)
    path = tmp_path / "ckpt.pth"
    torch.save({"args": args, "state_dict": sd}, path)
    return str(path)


def _cli_pair(tmp_path, ckpt, x, chunk_rows, nproc):
    np.save(tmp_path / "x.npy", x)
    common = ["--ckpt_path", ckpt, "--data_path", str(tmp_path / "x.npy"), "--dataset", "Toy", "--chunk_rows", str(chunk_rows)]
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        one = G.main(common + ["--output_dir", str(tmp_path / "one")])
    r = _torchrun("-m", "lcrec_b200.generate_indices", *common, "--output_dir", str(tmp_path / "many"), "--dist_timeout", "120",
                  nproc=nproc)
    assert r.returncode == 0, r.stderr[-3000:]
    many = tmp_path / "many" / "Toy.index.json"
    return open(one, "rb").read(), many.read_bytes(), _stat_lines(buf.getvalue()), _stat_lines(r.stdout)


DIMS = [96, 64, 32]
NPROC = 8 if N_GPUS >= 8 else 2


@multi_gpu
@pytest.mark.parametrize("case", ["fp32", "fp16", "one_item"])
def test_cli_sharded_equals_one_gpu(tmp_path, case):
    """fp32 / fp16 .npy of an odd N = 20 001 in chunks of 5000 rows (pieces on both RQ paths); N = 1 leaves ranks empty."""
    ckpt = _checkpoint(tmp_path, [256] * 4, DIMS)
    n = 1 if case == "one_item" else 20001
    x = synth_items(n, DIMS[0], n_parents=max(n // 6, 1), seed=21)
    if case == "fp16":
        x = x.astype(np.float16)
    one, many, s1, sn = _cli_pair(tmp_path, ckpt, x, 5000, NPROC)
    assert len(one) > 10 and many == one
    assert len(s1) == 3 and sn == s1


@multi_gpu
def test_cli_sharded_slab_overflow_falls_back_together(tmp_path):
    """Every item in buckets of rank 0: each rank's slab to rank 0 overflows (24 000 rows > 25 % slack + 4096); all ranks
    agree on it before the all-to-all and take the split-size path - no hang, the same bytes as one GPU."""
    ckpt = _checkpoint(tmp_path, [64, 256], DIMS, skew=True)
    n = 48000
    x = synth_items(n, DIMS[0], n_parents=n // 6, seed=22)
    one, many, s1, sn = _cli_pair(tmp_path, ckpt, x, 131072, NPROC)
    assert many == one and len(s1) == 3 and sn == s1
    codes = np.array([[int(t.split("_")[1][:-1]) for t in v] for v in json.loads(one).values()])
    cd = torch.from_numpy(codes)
    assert int((bucket_owner(cd, [64, 256], NPROC) == 0).sum()) == n      # the skew the case is about


def test_cli_torchrun_one_process_equals_plain_cli(tmp_path):
    ckpt = _checkpoint(tmp_path, [256] * 4, DIMS)
    x = synth_items(3001, DIMS[0], n_parents=500, seed=23)
    one, many, s1, sn = _cli_pair(tmp_path, ckpt, x, 1024, 1)
    assert many == one and len(s1) == 3 and sn == s1
