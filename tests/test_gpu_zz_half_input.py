"""Half-precision embeddings read natively (B200): fp16 / bf16 input through every layer that accepts it - the encoder
entry, the indexer on device and host input, PASS 0 in pieces, the CLI, the embedding producer and the sharded path -
against the fp32 path on the same values upcast with x.to(torch.float32).  Upcasting half to fp32 is exact, so every
comparison is bitwise (torch.equal), not a tolerance."""
import argparse
import os
import types

import numpy as np
import pytest
import torch

from tests.conftest import state_dict_of
from lcrec_b200.synth import seeded_weights, synth_items

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from lcrec_b200 import _lib, ops
    from lcrec_b200 import generate_indices as G
    from lcrec_b200.models import RQVAE
    DEV = torch.device("cuda:0")

HALVES = [torch.float16, torch.bfloat16]
RUNSH_DIMS = [4096, 2048, 1024, 512, 256, 128, 64, 32]


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def small_model(golden):
    g = golden("small_model")
    m = RQVAE(in_dim=96, num_emb_list=[32] * 4, e_dim=16, layers=[64, 48], sk_epsilons=[0.0, 0.0, 0.0, 0.003], sk_iters=50)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in state_dict_of(g).items()})
    return g, m.to(DEV).eval()


def runsh_model():
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


def forward_ex(h, x):
    """lcrec_mlp_forward_ex on x as it is (any dtype code, any base alignment)."""
    n = x.shape[0]
    y = torch.empty((n, h.dims[-1]), dtype=torch.float32, device=DEV)
    ws = ops._ws(h.lib.lcrec_mlp_workspace_bytes(h.handle, n), DEV)
    _lib.check(h.lib.lcrec_mlp_forward_ex(h.handle, ops._p(x), ops.DTYPE_CODES[x.dtype], n, ops._p(y), None, ops._p(ws),
                                          ws.numel(), ops._stream(x)))
    return y


def hostile_rows(n, k, dtype, seed):
    """n x k half rows: normal values, a row of zeros, and rows whose first 256-column group spans the subnormals of the
    format up to 2^15 with both signs (the split's group maximum, frexp scale and lo term at their extremes)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn((n, k), device=DEV, generator=g)
    if n > 1:
        x[1] = 0.0
    lo = -24 if dtype == torch.float16 else -133                 # smallest subnormal exponent of the format
    e = torch.linspace(lo, 15, min(256, k), device=DEV)
    span = torch.exp2(e) * (1 + 0.37 * torch.rand(e.shape, device=DEV, generator=g))
    span = torch.where(torch.arange(e.numel(), device=DEV) % 2 == 1, -span, span).clamp(-60000.0, 60000.0)
    for r in range(2, min(n, 6)):
        x[r, : e.numel()] = span.roll(r)
    return x.to(dtype)


# ------------------------------------------------------------------ 1. encoder
@pytest.fixture(scope="module")
def encoders():
    """the run.sh encoder (layer 1 on the CTA-pair kernel) and one whose layer 1 the pair kernel does not serve
    (n_out 96: single-CTA kernel with per-row scales; k = 200, not a multiple of 8)"""
    out = {}
    for name, dims in (("pair", RUNSH_DIMS), ("single", [200, 96, 64, 32])):
        ws, bs, _ = seeded_weights(dims, [8], dims[-1], seed=5)
        out[name] = ops.MlpHandle([T(w) for w in ws], [T(b) for b in bs])
    return out


@pytest.mark.parametrize("enc", ["pair", "single"])
@pytest.mark.parametrize("n_rows", [1, 33, 4097, 131073])
@pytest.mark.parametrize("dtype", HALVES, ids=["fp16", "bf16"])
def test_encoder_half_equals_fp32_upcast(encoders, enc, n_rows, dtype):
    h = encoders[enc]
    x = hostile_rows(n_rows, h.dims[0], dtype, seed=n_rows)
    want = h.forward(x.to(torch.float32))                       # lcrec_mlp_forward on the upcast input
    got = forward_ex(h, x)
    assert torch.isfinite(want).all()
    assert torch.equal(got, want)
    # a misaligned base (element offset 1: 2-byte aligned) takes the scalar loads
    flat = torch.empty(n_rows * h.dims[0] + 1, dtype=dtype, device=DEV)
    xm = flat[1:].view(n_rows, h.dims[0])
    xm.copy_(x)
    assert xm.data_ptr() % 8 != 0
    assert torch.equal(forward_ex(h, xm), want)


def test_encoder_engine0_refuses_half(encoders):
    """The tf32 x3 engine (cross-checks) has no half variant: a loud error naming the engine, never a conversion."""
    h = encoders["single"]
    x = hostile_rows(8, h.dims[0], torch.bfloat16, 1)
    try:
        h.set_engine(0)
        with pytest.raises(RuntimeError, match="engine 0"):
            forward_ex(h, x)
        x32 = x.to(torch.float32)
        assert torch.equal(forward_ex(h, x32), h.forward(x32))          # dtype 0 through the _ex entry is the fp32 entry
    finally:
        h.set_engine(1)


# ------------------------------------------------------------------ 2. indexer, device input
@pytest.mark.parametrize("dtype", HALVES, ids=["fp16", "bf16"])
def test_indexer_device_small_model(golden, dtype):
    g, m = small_model(golden)
    x = T(g["x"]).to(dtype)
    ix = G.build_indexer(m, x.shape[0])
    c_ref, s_ref = ix.run_device(x.to(torch.float32), 20)
    c, s = ix.run_device(x, 20)
    assert torch.equal(c, c_ref) and s == s_ref


@pytest.fixture(scope="module")
def runsh():
    return runsh_model()


@pytest.mark.parametrize("dtype", HALVES, ids=["fp16", "bf16"])
def test_indexer_device_several_chunks(runsh, dtype):
    """20 000 items in chunks of 4096 (five encoder calls, tensor-core RQ path), collision rounds included."""
    x = T(synth_items(20000, 4096, n_parents=2500, seed=11)).to(dtype)
    ix = G.build_indexer(runsh, x.shape[0], 4096)
    c_ref, s_ref = ix.run_device(x.to(torch.float32), 20)
    c, s = ix.run_device(x, 20)
    assert s_ref["rounds"] >= 2
    assert torch.equal(c, c_ref) and s == s_ref


# ------------------------------------------------------------------ 3. indexer, host input
@pytest.mark.parametrize("pinned", [True, False], ids=["pinned", "pageable"])
@pytest.mark.parametrize("dtype", HALVES, ids=["fp16", "bf16"])
def test_indexer_host_equals_device(runsh, dtype, pinned):
    """50 000 rows in chunks of 32 768: the last chunk (17 232 rows) is cut into two tail pieces."""
    n = 50000
    xd = T(synth_items(n, 4096, n_parents=n // 8, seed=12)).to(dtype)
    ix = G.build_indexer(runsh, n, 32768)
    c_dev, s_dev = ix.run_device(xd, 20)
    xh = xd.cpu()
    if pinned:
        xh = xh.pin_memory()
    c_host, s_host = ix.run_host(xh, max_rounds=20)
    assert not c_host.is_cuda and torch.equal(c_host, c_dev.cpu()) and s_host == s_dev
    c32, s32 = ix.run_device(xd.to(torch.float32), 20)
    assert torch.equal(c32, c_dev) and s32 == s_dev


# ------------------------------------------------------------------ 4. PASS 0 in pieces
@pytest.mark.parametrize("dtype", HALVES, ids=["fp16", "bf16"])
def test_pass0_row_offset_halves(runsh, dtype):
    n, half = 12000, 5000
    x = T(synth_items(n, 4096, n_parents=n // 8, seed=13)).to(dtype)
    ix = G.build_indexer(runsh, n, 4096)
    ix.pass0(x[:half], 0)
    ix.pass0(x[half:], half)
    codes, resid = ix.codes_view(n).clone(), ix.resid_view(n).clone()
    ix.pass0(x)
    assert torch.equal(codes, ix.codes_view(n)) and torch.equal(resid, ix.resid_view(n))
    ix.pass0(x.to(torch.float32))
    assert torch.equal(codes, ix.codes_view(n)) and torch.equal(resid, ix.resid_view(n))


# ------------------------------------------------------------------ 5. no fp32 copy
def test_run_device_makes_no_fp32_copy(runsh):
    n = 200000
    ix = G.build_indexer(runsh, n)
    x = torch.empty((n, 4096), dtype=torch.bfloat16, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(14)
    for s in range(0, n, 50000):
        x[s:s + 50000] = torch.randn((50000, 4096), device=DEV, generator=g)
    ix.run_device(x[:1000], 20)                                 # lazily created state outside the measurement
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(DEV)
    base = torch.cuda.memory_allocated(DEV)
    codes, _ = ix.run_device(x, 20)
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated(DEV) - base
    assert codes.shape == (n, 4)
    assert grown < n * 4096 * 4, grown                          # an fp32 copy of x alone would be 3.3 GB


# ------------------------------------------------------------------ 6. CLI on an fp16 .npy
def test_cli_fp16_npy_equals_fp32_npy(golden, tmp_path):
    g, m = small_model(golden)
    x16 = g["x"].astype(np.float16)
    np.save(tmp_path / "x16.npy", x16)
    np.save(tmp_path / "x32.npy", x16.astype(np.float32))
    args = argparse.Namespace(data_path=str(tmp_path / "x32.npy"), num_emb_list=[32] * 4, e_dim=16, layers=[64, 48],
                              dropout_prob=0.0, bn=False, loss_type="mse", quant_loss_weight=1.0, kmeans_init=False,
                              kmeans_iters=100, sk_epsilons=[0.0, 0.0, 0.0, 0.003], sk_iters=50)
    torch.save({"args": args, "state_dict": {k: v.cpu() for k, v in m.state_dict().items()}}, tmp_path / "ckpt.pth")
    out = {}
    for tag in ("x16", "x32"):
        path = G.main(["--ckpt_path", str(tmp_path / "ckpt.pth"), "--output_dir", str(tmp_path / tag), "--dataset", "Toy",
                       "--data_path", str(tmp_path / f"{tag}.npy"), "--chunk_rows", "512"])
        out[tag] = open(path, "rb").read()
    assert len(out["x16"]) > 1000 and out["x16"] == out["x32"]


# ------------------------------------------------------------------ 7. producer
class _Encoded(dict):
    def to(self, device):
        return _Encoded({k: v.to(device) for k, v in self.items()})
    input_ids = property(lambda self: self["input_ids"])
    attention_mask = property(lambda self: self["attention_mask"])


def _standins(hidden=200, vocab=50, seq=12):
    gen = torch.Generator().manual_seed(3)
    E = torch.randn((vocab, hidden), generator=gen).to(DEV)

    def tokenizer(sentences, max_length, truncation, return_tensors, padding):
        items = [int(s.split()[1]) for s in sentences]
        lens = [1 + (7 * i + len(s)) % seq for i, s in zip(items, sentences)]
        t = max(lens)
        ids = torch.tensor([[(3 * i + j + len(s)) % vocab for j in range(t)] for i, s in zip(items, sentences)])
        mask = torch.tensor([[1 if j < l else 0 for j in range(t)] for l in lens])
        return _Encoded(input_ids=ids, attention_mask=mask)

    def model(input_ids, attention_mask):
        return types.SimpleNamespace(last_hidden_state=E[input_ids] * (1 + input_ids[..., None] % 5))

    return tokenizer, model


@pytest.mark.parametrize("dtype", HALVES, ids=["fp16", "bf16"])
def test_producer_half_matrix(tmp_path, dtype):
    from lcrec_b200.text_emb import generate_item_embedding
    tokenizer, model = _standins()
    items = [[i, ["title %d" % i, "description %d long" % i]] for i in reversed(range(10))]
    args = types.SimpleNamespace(root=str(tmp_path), dataset="Toy", plm_name="standin", max_sent_len=24, device=DEV)
    ref = generate_item_embedding(args, items, tokenizer, model, batch_size=3, save=False)
    save = dtype == torch.float16
    emb = generate_item_embedding(args, items, tokenizer, model, batch_size=3, save=save, dtype=dtype)
    assert ref.dtype == torch.float32 and emb.dtype == dtype and emb.is_cuda
    assert torch.equal(emb, ref.to(dtype))
    if save:
        saved = np.load(os.path.join(str(tmp_path), "Toy.emb-standin-td.npy"))
        assert saved.dtype == np.float16 and np.array_equal(saved, emb.cpu().numpy())
    else:
        with pytest.raises(ValueError, match="bfloat16"):
            generate_item_embedding(args, items, tokenizer, model, batch_size=3, save=True, dtype=dtype)


# ------------------------------------------------------------------ 8. engine 0 through the indexer
def test_indexer_engine0_refuses_half(golden):
    g, m = small_model(golden)
    ix = G.build_indexer(m, int(g["x"].shape[0]))
    try:
        ix.encoder.set_engine(0)
        with pytest.raises(RuntimeError, match="engine 0"):
            ix.run_device(T(g["x"]).to(torch.bfloat16), 20)
    finally:
        ix.encoder.set_engine(ops.DEFAULT_ENGINE)


# ------------------------------------------------------------------ 9. two GPUs
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_bf16_equals_single_gpu():
    """2 ranks from bf16 shards (all-to-all bucket exchange + native rounds per owner) == one GPU over the bf16 union."""
    import json, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29579", os.path.join(root, "scripts", "check_sharded_equals_single.py"),
                        "200003", "bfloat16"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["ok"] and out["identical"] and out["dtype"] == "bfloat16"
