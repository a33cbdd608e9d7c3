"""torchrun --nproc-per-node N scripts/check_dp_ema.py : data-parallel training of the EMA-codebook variant (index_improve).

* op level: ``DistributedEma.update`` on every rank == ``ops.ema_update`` on the concatenated global batch on that rank's GPU
  and == ``oracle.ema_update``, bit for bit; replicas compared whole (MIN / MAX all-reduces); consecutive calls on one
  instance that alternate levels and shapes (both slots reused); a block over capacity or other than the rank's ShardPlan
  share raises ValueError before any device work;
* the dead-code reset over the global batch == single-device ``_reset_unused_codes`` under the same seed on rank 0;
* ``index_improve.trainer.DataParallelTrainer`` against the unmodified reference Trainer (tests/golden/ema_trainer_steps.npz),
  replicas, the first step bitwise against the single-device trainer, resets during training, an empty rank, the k-means
  pass, BatchNorm;
* ms per step at the run.sh shape (global batch 1024), EMA variant against the plain one, alternated, and CUDA-event
  times of the per-level EMA step (``--no-timing`` skips this part).
Prints one JSON line on rank 0."""
import argparse, json, os, subprocess, sys, tempfile, time
import numpy as np
import torch, torch.distributed as dist
root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, root)
from lcrec_b200 import ops
from lcrec_b200.distributed import DistributedEma, ShardPlan
from lcrec_b200.index_improve.models import RQVAE, VectorQuantizer
from lcrec_b200.index_improve.trainer import DataParallelTrainer, Trainer
from oracle import lcrec_oracle as O

cli = argparse.ArgumentParser()
cli.add_argument("--no-timing", action="store_true")
opts = cli.parse_args()
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
dev = torch.device(f"cuda:{local}")
torch.cuda.set_device(dev)
dist.init_process_group("nccl", device_id=dev)
failures = []


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def same_on_all_ranks(tensors):
    """Every tensor bit-identical on every rank: MIN and MAX of the whole flattened state (fp32 / int64 -> fp64 is exact for
    the values compared here; int64 buffers are small counters)."""
    flat = torch.cat([t.detach().reshape(-1).double() for t in tensors]) if tensors else torch.zeros(1, device=dev, dtype=torch.float64)
    nan = torch.isnan(flat).any().to(torch.float64).reshape(1)
    flat = torch.nan_to_num(flat, nan=1.2345e300)
    lo, hi = flat.clone(), flat.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    dist.all_reduce(nan, op=dist.ReduceOp.MAX)
    return bool(torch.equal(lo, hi)) and not bool(nan.item())


def all_ranks(flag):
    t = torch.tensor([1 if flag else 0], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return bool(t.item())


def check(name, ok):
    ok = all_ranks(ok)
    if not ok:
        failures.append(name)
    return ok


# ---------------------------------------------------------------------------------------------------------------- op level
def ema_case(n, k, d, skew, steps, dema=None, st=None, seed=None):
    """`steps` EMA steps of one level over a global batch of n rows split by ShardPlan; returns (ok, state)."""
    rng = np.random.default_rng(seed if seed is not None else n + 31 * k + d)
    if st is None:
        st = O.EmaState((rng.standard_normal((k, d)) * 0.05).astype(np.float32),
                        (rng.random(k) * (rng.random(k) < 0.7)).astype(np.float32),
                        (rng.standard_normal((k, d)) * 0.01).astype(np.float32))
    cb, cs, w = T(st.codebook), T(st.cluster_size), T(st.ema_w)          # distributed
    cb1, cs1, w1 = cb.clone(), cs.clone(), w.clone()                      # single device, this rank's GPU
    if dema is None:
        dema = DistributedEma(max(1, ShardPlan(n, world).max_count), d, dev)
    plan = ShardPlan(n, world)
    ok = True
    for _ in range(steps):
        x = (rng.standard_normal((n, d)) * 0.1).astype(np.float32)
        idx = rng.integers(0, k, size=n)
        idx = np.where(rng.random(n) < skew, 3 % k, idx).astype(np.int64)
        st = O.ema_update(x, idx, st, 0.99, 1e-5)
        sl = plan.slice(rank)
        glat = dema.update(T(x[sl]), T(idx[sl]), n, cs, w, cb, 0.99, 1e-5)
        ops.ema_update(T(x), T(idx), cs1, w1, cb1, 0.99, 1e-5)
        ok &= torch.equal(glat, T(x)) and torch.equal(dema.gathered_indices[:n], T(idx))
        ok &= torch.equal(cs, cs1) and torch.equal(w, w1) and torch.equal(cb, cb1)
        ok &= np.array_equal(cs.cpu().numpy(), st.cluster_size) and np.array_equal(w.cpu().numpy(), st.ema_w)
        ok &= np.array_equal(cb.cpu().numpy(), st.codebook)
        ok &= same_on_all_ranks([cs, w, cb])
    return ok, st


op_cases = {}
with ops.defer_checks():
    for (n, k, d, skew) in [(1, 4, 8, 0.0), (0, 8, 4, 0.0), (257, 32, 16, 0.0), (5000, 256, 32, 0.8), (4097, 300, 100, 0.5),
                            (2000, 8192, 256, 0.0)]:
        ok, _ = ema_case(n, k, d, skew, steps=2)
        op_cases[f"{n}x{k}x{d}"] = check(f"op {n}x{k}x{d}", ok)
    ops.flush_checks()

    # consecutive calls on ONE instance: 4 levels of different K, row counts 0 / 1 / ragged / full, 12 calls
    cap = ShardPlan(1200, world).max_count
    dema = DistributedEma(cap, 32, dev)
    states = [None] * 4
    ok = True
    for c, n in enumerate([1000, 1, 0, 1199, 257, 1200, 3, 999, 64, 1000, 2, 555]):
        lvl = c % 4
        good, states[lvl] = ema_case(n, [256, 64, 256, 17][lvl], 32, 0.3 if lvl == 1 else 0.0, 1, dema=dema, st=states[lvl],
                                     seed=1000 + c)
        ok &= good
    op_cases["consecutive_calls_one_instance"] = check("consecutive calls", ok and dema.epoch == 12)
    ops.flush_checks()
    try:                                                   # one row too many: rank 0's block exceeds the capacity
        n_over = world * cap + 1
        m_over = ShardPlan(n_over, world).count(rank)
        dema.update(torch.zeros((m_over, 32), device=dev), torch.zeros(m_over, dtype=torch.int64, device=dev), n_over,
                    torch.zeros(8, device=dev), torch.zeros(8, 32, device=dev), torch.zeros(8, 32, device=dev), 0.99, 1e-5)
        raised = False
    except ValueError:
        raised = True
    op_cases["over_capacity_raises_everywhere"] = check("over capacity", raised and dema.epoch == 12)
    try:                                                   # every rank passes 1 row where its ShardPlan share is 2
        dema.update(torch.zeros((1, 32), device=dev), torch.zeros(1, dtype=torch.int64, device=dev), 2 * world,
                    torch.zeros(8, device=dev), torch.zeros(8, 32, device=dev), torch.zeros(8, 32, device=dev), 0.99, 1e-5)
        raised = False
    except ValueError:
        raised = True
    op_cases["wrong_share_raises_everywhere"] = check("wrong share", raised and dema.epoch == 12)

# ---------------------------------------------------------------------------------------------------------------- reset
gk = dict(np.load(os.path.join(root, "tests", "golden", "ema_kat.npz")))
n_e, e_dim, _, batch = (int(v) for v in gk["c2_cfg"])
x = T(gk["c2_s2_x"])


def level():
    vq = VectorQuantizer(n_e, e_dim, sk_epsilon=0.0, reset_interval=3).to(dev).train()
    vq.embedding.weight.data.copy_(T(gk["c2_s2_pre_reset_codebook"]))
    vq._ema_cluster_size.copy_(T(gk["c2_s2_pre_reset_cs"]))
    vq._ema_w.fill_(1.0)
    return vq


ref = level()
torch.manual_seed(7)
ref._reset_unused_codes(x)
vq = level()
vq.dist_ema = DistributedEma(ShardPlan(batch, world).max_count, e_dim, dev)
with ops.defer_checks():                                   # the gathered latent: an update on throw-away buffers
    glat = vq.dist_ema.update(x[ShardPlan(batch, world).slice(rank)], torch.zeros(ShardPlan(batch, world).count(rank), dtype=torch.int64, device=dev),
                              batch, torch.zeros(n_e, device=dev), torch.zeros(n_e, e_dim, device=dev),
                              torch.zeros(n_e, e_dim, device=dev), 0.99, 1e-5)
    ops.flush_checks()
torch.manual_seed(7 if rank == 0 else 1000 + rank)          # only rank 0's RNG may matter
vq._reset_unused_codes_dist(glat)
reset_ok = check("reset", torch.equal(glat, x) and torch.equal(vq.embedding.weight, ref.embedding.weight)
                 and torch.equal(vq._ema_cluster_size, ref._ema_cluster_size) and torch.equal(vq._ema_w, ref._ema_w)
                 and same_on_all_ranks([vq.embedding.weight, vq._ema_cluster_size, vq._ema_w])
                 and not torch.equal(ref.embedding.weight, T(gk["c2_s2_pre_reset_codebook"])))

# ---------------------------------------------------------------------------------------------------------------- trainer
g = dict(np.load(os.path.join(root, "tests", "golden", "ema_trainer_steps.npz")))


def make_args(**kw):
    base = dict(lr=1e-3, epochs=4, batch_size=256, num_workers=0, eval_step=50, learner="AdamW", lr_scheduler_type="linear",
                warmup_epochs=1, data_path="", weight_decay=1e-4, dropout_prob=0.0, bn=False, loss_type="mse", kmeans_init=False,
                kmeans_iters=10, sk_epsilons=[0.0, 0.0, 0.0, 0.003], sk_iters=50, device=str(dev), num_emb_list=[32] * 4, e_dim=16,
                quant_loss_weight=1.0, beta=0.25, layers=[64, 48], save_limit=5, ckpt_dir=tempfile.mkdtemp(prefix="dp_ema_ckpt_"),
                ema_decay=0.99, epsilon=1e-5, reset_threshold=1e-5, reset_interval=1000)
    base.update(kw)
    return argparse.Namespace(**base)


def make_model(args, golden_init=True, seed=0):
    torch.manual_seed(seed)
    m = RQVAE(in_dim=96, num_emb_list=args.num_emb_list, e_dim=args.e_dim, layers=args.layers, bn=args.bn,
              kmeans_init=args.kmeans_init, kmeans_iters=args.kmeans_iters, sk_epsilons=args.sk_epsilons, sk_iters=args.sk_iters,
              ema_decay=args.ema_decay, epsilon=args.epsilon, reset_threshold=args.reset_threshold,
              reset_interval=args.reset_interval)
    if golden_init:
        m.load_state_dict({k[5:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("init/")})
    return m


def model_state(m):
    return [p.detach() for p in m.parameters()] + [b for b in m.buffers()] + \
        [torch.tensor([q.step_count for q in m.rq.vq_layers], device=dev)]


def ema_buffers(m):
    return [t for q in m.rq.vq_layers for t in (q._ema_cluster_size, q._ema_w, q.embedding.weight.detach())]


def loader_of(x, bs=256):
    return torch.utils.data.DataLoader(torch.from_numpy(x), batch_size=bs, shuffle=False)


trainer = {}
# the reference's bars (test_improve_trainer_matches_reference_losses)
args = make_args()
m = make_model(args)
loader = loader_of(g["x"])
tr = DataParallelTrainer(args, m, len(loader))
losses = np.array([tr._train_epoch(loader, ep) for ep in range(4)])
rel = float(np.abs(losses / g["losses"] - 1).max())
coll = tr._valid_epoch(loader)
avg, stats = tr._get_codebook_utilization()
used = [int(s["used_codes"]) for s in stats]
trainer["reference"] = {"max_rel_loss": rel, "collision_rate": coll, "reference_collision_rate": float(g["collision_rate"]),
                        "avg_utilization": float(avg), "reference_avg_utilization": float(g["avg_utilization"]),
                        "used_codes": used, "reference_used_codes": [int(u) for u in g["used_codes"]],
                        "step_counts": [q.step_count for q in m.rq.vq_layers]}
trainer["reference"]["ok"] = check("trainer reference bars", rel < 2e-3 and abs(coll - float(g["collision_rate"])) < 0.02
                                   and abs(avg - float(g["avg_utilization"])) <= 0.05
                                   and all(abs(a - int(b)) <= 2 for a, b in zip(used, g["used_codes"]))
                                   and all(q.step_count == 16 for q in m.rq.vq_layers))
trainer["replicas_equal"] = check("trainer replicas", same_on_all_ranks(model_state(m)))
del tr, m

# first step, bitwise against the single-device EMA trainer on the same global batch (sk 0, bn False)
args = make_args(sk_epsilons=[0.0] * 4, epochs=1)
m_dp, m_1 = make_model(args), make_model(args)
one = loader_of(g["x"][:256])
DataParallelTrainer(args, m_dp, 1)._train_epoch(one, 0)
Trainer(make_args(sk_epsilons=[0.0] * 4, epochs=1), m_1, 1)._train_epoch(one, 0)
trainer["first_step_ema_buffers_bitwise"] = check("first step bitwise", all(torch.equal(a, b) for a, b in zip(ema_buffers(m_dp), ema_buffers(m_1))))

# resets during training (reset_interval 3): count the codes the single-device run resets, replicas through the resets
args = make_args(reset_interval=3, epochs=2)
resets = []


def counting(q):
    orig = q._reset_unused_codes

    def wrapped(latent):
        _, mask = ops.codebook_usage(q._ema_cluster_size, q.epsilon, q.reset_threshold, want_unused=True)
        resets.append(min(int(mask.sum().item()), len(latent)))
        return orig(latent)
    q._reset_unused_codes = wrapped


m_1 = make_model(args)
for q in m_1.rq.vq_layers:
    counting(q)
tr1 = Trainer(args, m_1, len(loader))
single_losses = np.array([tr1._train_epoch(loader, ep) for ep in range(2)])
single_resets = sum(resets)
m_dp = make_model(args)
tr = DataParallelTrainer(args, m_dp, len(loader))
dp_losses = np.array([tr._train_epoch(loader, ep) for ep in range(2)])
trainer["reset_interval_3"] = {"codes_reset_single_device": single_resets,
                               "max_rel_loss_vs_single_device": float(np.abs(dp_losses / single_losses - 1).max()),
                               "replicas_equal": same_on_all_ranks(model_state(m_dp)),
                               "step_counts": [q.step_count for q in m_dp.rq.vq_layers]}
trainer["reset_interval_3"]["ok"] = check("resets", single_resets > 0 and trainer["reset_interval_3"]["replicas_equal"]
                                          and all(q.step_count == 8 for q in m_dp.rq.vq_layers))
del tr, tr1

# a final batch of one row leaves rank 1 empty; the reset is due on that very step (reset_interval 4)
args = make_args(reset_interval=4, epochs=1)
m_dp = make_model(args)
ragged = loader_of(g["x"][:3 * 256 + 1])
tr = DataParallelTrainer(args, m_dp, len(ragged))
tr._train_epoch(ragged, 0)
trainer["empty_rank"] = {"step_counts": [q.step_count for q in m_dp.rq.vq_layers], "replicas_equal": same_on_all_ranks(model_state(m_dp))}
trainer["empty_rank"]["ok"] = check("empty rank", trainer["empty_rank"]["replicas_equal"] and all(q.step_count == 4 for q in m_dp.rq.vq_layers))
del tr

# k-means pass: no EMA step in it
args = make_args(kmeans_init=True, epochs=1)
m_dp = make_model(args, golden_init=False)
DataParallelTrainer(args, m_dp, 1)._train_epoch(one, 0)
sums = [float(q._ema_cluster_size.double().sum()) for q in m_dp.rq.vq_layers]
trainer["kmeans_init"] = {"step_counts": [q.step_count for q in m_dp.rq.vq_layers], "cluster_size_sums": sums,
                          "want": (1 - 0.99) * 256, "replicas_equal": same_on_all_ranks(model_state(m_dp))}
trainer["kmeans_init"]["ok"] = check("kmeans init", all(q.step_count == 1 for q in m_dp.rq.vq_layers)
                                     and all(abs(s - (1 - 0.99) * 256) <= 1e-5 * 256 for s in sums)
                                     and trainer["kmeans_init"]["replicas_equal"])

# synchronised BatchNorm with the EMA levels
args = make_args(bn=True, epochs=2)
m_1, m_dp = make_model(args, golden_init=False, seed=3), make_model(args, golden_init=False, seed=3)
tr1 = Trainer(args, m_1, len(loader))
single_losses = np.array([tr1._train_epoch(loader, ep) for ep in range(2)])
tr = DataParallelTrainer(make_args(bn=True, epochs=2), m_dp, len(loader))
dp_losses = np.array([tr._train_epoch(loader, ep) for ep in range(2)])
bn_rel = float(np.abs(dp_losses / single_losses - 1).max())
trainer["batchnorm"] = {"max_rel_loss_vs_single_device": bn_rel, "replicas_equal": same_on_all_ranks(model_state(m_dp))}
trainer["batchnorm"]["ok"] = check("batchnorm", bn_rel < 2e-3 and trainer["batchnorm"]["replicas_equal"])
del tr, tr1

# ---------------------------------------------------------------------------------------------------------------- timing
timing = None
if not opts.no_timing:
    from lcrec_b200.dp_trainer import DataParallelTrainer as PlainDP
    from lcrec_b200.models import RQVAE as PlainRQVAE
    dims = [2048, 1024, 512, 256, 128, 64]
    targs = make_args(layers=dims, num_emb_list=[256] * 4, e_dim=32, epochs=1, batch_size=1024)
    xb = torch.randn(8 * 1024, 4096, generator=torch.Generator().manual_seed(1))
    tl = torch.utils.data.DataLoader(xb, batch_size=1024, shuffle=False)
    torch.manual_seed(0)
    mp = PlainRQVAE(in_dim=4096, num_emb_list=[256] * 4, e_dim=32, layers=dims, sk_epsilons=[0.0, 0.0, 0.0, 0.003], sk_iters=50)
    torch.manual_seed(0)
    me = RQVAE(in_dim=4096, num_emb_list=[256] * 4, e_dim=32, layers=dims, sk_epsilons=[0.0, 0.0, 0.0, 0.003], sk_iters=50)
    runs = {"plain": PlainDP(targs, mp, len(tl)), "ema": DataParallelTrainer(targs, me, len(tl))}
    for t in runs.values():
        t._train_epoch(tl, 0)                                            # warm-up
    ms = {k: [] for k in runs}
    for rep in range(4):                                                 # alternated in the same call
        for name, t in runs.items():
            torch.cuda.synchronize(); dist.barrier(); t0 = time.perf_counter()
            t._train_epoch(tl, 1 + rep)
            torch.cuda.synchronize(); dist.barrier()
            ms[name].append((time.perf_counter() - t0) / len(tl) * 1e3)
    # one level's EMA step at this shape: the three launches (CUDA events over 200 calls) against the third alone
    plan = ShardPlan(1024, world)
    de = runs["ema"]._ema
    lat = torch.randn(plan.count(rank), 32, device=dev)
    idx = torch.randint(0, 256, (plan.count(rank),), device=dev)
    cs, w, cb = torch.zeros(256, device=dev), torch.zeros(256, 32, device=dev), torch.randn(256, 32, device=dev)
    de.n_rows_hint = 1024
    glat = de.update(lat, idx, 1024, cs, w, cb, 0.99, 1e-5)
    gl, gi = glat.clone(), de.gathered_indices[:1024].clone()

    def events(fn, reps=200):
        fn()
        torch.cuda.synchronize(); dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record(); torch.cuda.synchronize()
        return a.elapsed_time(b) / reps * 1e3
    with ops.defer_checks():
        us_dist = events(lambda: de.update(lat, idx, 1024, cs, w, cb, 0.99, 1e-5))
        ops.flush_checks()
    us_kernel = events(lambda: ops.ema_update(gl, gi, cs, w, cb, 0.99, 1e-5))
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local)],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:                                               # the card name below still identifies the GPU
        smi = f"nvidia-smi unavailable: {e}"
    timing = {"card": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit": smi,
              "ms_per_step_plain": ms["plain"], "ms_per_step_ema": ms["ema"],
              "median_ms_plain": float(np.median(ms["plain"])), "median_ms_ema": float(np.median(ms["ema"])),
              "ema_level_us_three_launches": us_dist, "ema_level_us_ema_kernel_alone": us_kernel,
              "ema_level_us_publish_plus_gather": us_dist - us_kernel}

ok = not failures
if rank == 0:
    print(json.dumps({"world": world, "ok": ok, "failures": failures, "op_cases": op_cases, "reset": reset_ok,
                      "trainer": trainer, "timing": timing}))
dist.barrier()
dist.destroy_process_group()
