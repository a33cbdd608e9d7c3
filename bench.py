#!/usr/bin/env python
"""Benchmark of the LC-Rec item-indexing hot path on B200 (metric of BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # CPU arm: the reference algorithm on host cores
    python bench.py --steps K --warmup W --dump-outputs DIR   # + DIR/codes.npy: the codes of the last timed step

A step = one full pass of index generation (generate_indices.py:85-128: encoder -> 4-level residual
quantisation -> up to 20 rounds of sort/unique + per-group Sinkhorn) over the whole synthetic item set.
Workload (BASELINE.json configs[2], the largest that fits one GPU): 1 M items x 4096-d fp32 per GPU,
encoder 4096-2048-1024-512-256-128-64-32, 4 x 256 codes, e_dim 32, eps_last 0.003, 50 Sinkhorn
iterations; for N > 1 every rank holds its own 1 M items (weak scaling, BASELINE.json configs[3] shape)
and the ranks resolve collisions over the union (one all-gather of codes + residuals, prefix-bucket ownership,
one all-reduce of the final last-level codes; NCCL).
Inputs (16.4 GB per GPU) are larger than the 126 MB L2, so no flush is needed between steps.
One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DIMS = [4096, 2048, 1024, 512, 256, 128, 64, 32]
N_CODES = [256, 256, 256, 256]
E_DIM = 32
EPS_LAST = 0.003
SK_ITERS = 50
SEED_W = 77
SEED_X = 2024
HEAD_ITEMS = 8192          # numpy-generated head of the item stream, shared with the CPU arm
BYTES_PER_ITEM = DIMS[0] * 4 + len(N_CODES) * 8                       # 16 416 B (SURVEY 8(d))
FLOP_PER_ITEM = 2 * sum(a * b for a, b in zip(DIMS[:-1], DIMS[1:])) + len(N_CODES) * 2 * 256 * E_DIM   # 22 433 792


def set_config(name):
    """c3 (default; BASELINE configs[2] / [3]): 4 x 256 codes, e_dim 32.  c5 (configs[4]): 4 x 8192 codes, e_dim 256 (encoder tail
    64 -> 256; tensor-core distance GEMM path).  c2 (configs[1]) is the training epoch: run_c2()."""
    global DIMS, N_CODES, E_DIM, BYTES_PER_ITEM, FLOP_PER_ITEM, CONFIG
    CONFIG = name
    if name == "c5":
        DIMS = [4096, 2048, 1024, 512, 256, 128, 64, 256]
        N_CODES = [8192] * 4
        E_DIM = 256
    BYTES_PER_ITEM = DIMS[0] * 4 + len(N_CODES) * 8
    FLOP_PER_ITEM = 2 * sum(a * b for a, b in zip(DIMS[:-1], DIMS[1:])) + sum(2 * k * E_DIM for k in N_CODES)


CONFIG = "c3"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_burst": d["bf16_tflops"], "bf16_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_burst": 1590.0, "bf16_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


# ----------------------------------------------------------------------------- workload (numpy, shared by both arms)
def np_mlp(x, ws, bs):
    h = x
    for i, (w, b) in enumerate(zip(ws, bs)):
        h = h @ w.T + b
        if i != len(ws) - 1:
            h = np.maximum(h, 0)
    return h.astype(np.float32)


def make_model():
    """Seeded encoder weights + data-driven codebooks (sample init + 4 Lloyd steps per level on the
    latents of the stream head).  Pure numpy so that the CPU arm and the GPU arm hold identical parameters."""
    from lcrec_b200.synth import seeded_weights, synth_items
    ws, bs, _ = seeded_weights(DIMS, N_CODES, E_DIM, seed=SEED_W)
    head = synth_items(HEAD_ITEMS, DIMS[0], n_parents=HEAD_ITEMS // 8, seed=SEED_X)
    z = np_mlp(head, ws, bs)
    rng = np.random.default_rng(5)
    resid = z.copy()
    cbs = []
    for k in N_CODES:
        if k * 4 > resid.shape[0]:          # large codebooks (c5): residual rows + a little noise, no Lloyd steps
            cb = resid[rng.integers(0, resid.shape[0], size=k)] + np.float32(1e-3 * resid.std()) * rng.standard_normal((k, resid.shape[1]), dtype=np.float32)
            d = (resid ** 2).sum(1, keepdims=True) + (cb ** 2).sum(1)[None] - 2 * resid @ cb.T
            resid = resid - cb[d.argmin(1)]
            cbs.append(cb.astype(np.float32))
            continue
        cb = resid[rng.choice(resid.shape[0], k, replace=False)].copy()
        for _ in range(4):
            d = (resid ** 2).sum(1, keepdims=True) + (cb ** 2).sum(1)[None] - 2 * resid @ cb.T
            a = d.argmin(1)
            for c in range(k):
                m = a == c
                if m.any():
                    cb[c] = resid[m].mean(0)
        d = (resid ** 2).sum(1, keepdims=True) + (cb ** 2).sum(1)[None] - 2 * resid @ cb.T
        resid = resid - cb[d.argmin(1)]
        cbs.append(cb.astype(np.float32))
    return ws, bs, cbs, head


def make_items_device(n, head, device, rank):
    """n items on the device: the numpy head first, the rest from the same generator family with the
    torch device RNG (low-rank parents + 0.05 noise, ~8 near-duplicates per parent)."""
    import torch
    from lcrec_b200.synth import lowrank_map, RANK
    x = torch.empty((n, DIMS[0]), dtype=torch.float32, device=device)
    h = min(n, head.shape[0]) if rank == 0 else 0
    if h:
        x[:h] = torch.from_numpy(head[:h]).to(device)
    g = torch.Generator(device=device).manual_seed(SEED_X + 1000 * rank)
    gmap = torch.from_numpy(lowrank_map(DIMS[0])).to(device)
    n_par = max((n - h) // 8, 1)
    parents = torch.randn((n_par, RANK), device=device, generator=g)
    for s in range(h, n, 65536):
        m = min(65536, n - s)
        pid = torch.randint(0, n_par, (m,), device=device, generator=g)
        x[s:s + m] = parents[pid] @ gmap
        x[s:s + m].add_(torch.randn((m, DIMS[0]), device=device, generator=g), alpha=0.05)
    return x


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.path = tempfile.mktemp(prefix="lcrec_clocks_", suffix=".csv")
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "25"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:  # noqa: BLE001
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [t.strip() for t in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        try:
            os.remove(self.path)
        except OSError:
            pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "power_w_max": float(max(power)), "samples": len(sm)}


# ----------------------------------------------------------------------------- CPU arm
REF_ITEM_RUNS = 150_000      # item-runs the reference arm may spend in total (~4 min at the ~600 items/s of the round-1 box)
C1_ITEMS = 25_000            # BASELINE.json configs[0]


def reference_sample_items(steps, warmup):
    """Items per step of the reference arm: C1 in full (25 000) when steps + warmup <= 6, otherwise the largest sample that
    keeps the whole `--steps K --warmup W` run within a few minutes.  A pure function of (K, W) so that both arms print it."""
    return int(min(C1_ITEMS, max(2048, REF_ITEM_RUNS // max(steps + warmup, 1))))


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        return os.cpu_count() or 1


def reference_items(n):
    from lcrec_b200.synth import synth_items
    return synth_items(n, DIMS[0], n_parents=max(n // 8, 1), seed=SEED_X)


def run_reference_script(ws, bs, cbs, x, device, repeat, threads, timeout_s=1500):
    """baseline/run_reference.py in a subprocess: the UNMODIFIED index/generate_indices.py (staged under baseline/_ref by
    build()) on x.  torchrun exports OMP_NUM_THREADS=1; the thread count is set explicitly here.  Returns the runner's dict
    (seconds per repeat, torch threads, ...) or {"unavailable": why}."""
    runner = os.path.join(ROOT, "baseline", "run_reference.py")
    if not os.path.isfile(os.path.join(ROOT, "baseline", "_ref", "index", "generate_indices.py")):
        return {"unavailable": "baseline/_ref/index not staged"}
    tmp = tempfile.mkdtemp(prefix="lcrec_refarm_")
    npz = os.path.join(tmp, "in.npz")
    arrs = {"x": x, "eps": np.array([0.0, 0.0, 0.0, EPS_LAST]), "sk_iters": np.int64(SK_ITERS)}
    for i, (w, b) in enumerate(zip(ws, bs)):
        arrs[f"w{i}"] = w; arrs[f"b{i}"] = b
    for l, cb in enumerate(cbs):
        arrs[f"cb{l}"] = cb
    np.savez(npz, **arrs)
    env = dict(os.environ)
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
        env[k] = str(threads)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "PYTHONPATH"):
        env.pop(k, None)
    out = os.path.join(tmp, "out.json")
    try:
        r = subprocess.run([sys.executable, runner, "--npz", npz, "--device", device, "--threads", str(threads), "--repeat", str(repeat),
                            "--out", out], env=env, cwd=tmp, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=timeout_s)
        if r.returncode != 0 or not os.path.exists(out):
            return {"unavailable": f"runner exit {r.returncode}: {r.stderr.strip()[-300:]}"}
        return json.load(open(out))
    except subprocess.TimeoutExpired:
        return {"unavailable": f"runner exceeded {timeout_s} s"}
    finally:
        for f in (npz, out):
            try:
                os.remove(f)
            except OSError:
                pass


def cpu_port_run(ws, bs, cbs, x):
    """Fallback when baseline/_ref is not staged: the numpy restatement (oracle), literal per-group re-encoding."""
    from oracle import lcrec_oracle as O
    p = O.RqvaeParams(encoder=O.MlpParams(ws, bs), codebooks=cbs, sk_epsilons=[0.0, 0.0, 0.0, EPS_LAST], sk_iters=SK_ITERS)
    t0 = time.perf_counter()
    O.generate_indices(x, p, batch_size=64, max_rounds=20, reencode=True)
    return time.perf_counter() - t0


def cpu_baseline(ws, bs, cbs, n_items, repeat=1, drop=0):
    """(dict for the JSON line, mean seconds per run).  kind "reference" = the unmodified script on torch-CPU."""
    x = reference_items(n_items)
    cores = host_cores()
    res = run_reference_script(ws, bs, cbs, x, "cpu", repeat, cores)
    if "unavailable" not in res:
        secs = res["seconds"][drop:]
        dt = float(np.mean(secs))
        return {"value": n_items / dt, "unit": "items/s", "cores": int(res["torch_threads"]), "kind": "reference", "seconds": dt,
                "host_cpus": res["cpu_count"], "torch": res["torch"], "rounds": res["rounds"],
                "collision_rate_final": res["collision_rate_final"],
                "sample": f"{n_items} items of the same synthetic stream per run: the UNMODIFIED index/generate_indices.py (baseline/_ref, "
                          f"torch CPU, DataLoader batch 64, per-group re-encoding, JSON dump), {len(secs)} timed run(s)"}, dt
    secs = [cpu_port_run(ws, bs, cbs, x) for _ in range(repeat)][drop:]
    dt = float(np.mean(secs))
    return {"value": n_items / dt, "unit": "items/s", "cores": cores, "kind": "port", "seconds": dt,
            "sample": f"{n_items} items, numpy restatement of generate_indices.py (oracle; {res['unavailable']})"}, dt


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    ws, bs, cbs, _ = make_model()
    n_sample = a.cpu_sample or reference_sample_items(a.steps, a.warmup)
    cpu, dt = cpu_baseline(ws, bs, cbs, n_sample, repeat=a.warmup + a.steps, drop=a.warmup)
    value = cpu["value"]
    line = {"impl": "reference", "metric": "items indexed/sec (4-level RQ + Sinkhorn collision resolution)", "value": value,
            "unit": "items/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(a.gpus, a.items, a.steps, a.warmup, a.cpu_sample),
            "cpu_baseline": cpu,
            "e2e": {"value": value, "unit": "items/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)
    return 0


def workload_config(gpus, items, steps, warmup, cpu_sample=None):
    n_ref = cpu_sample or reference_sample_items(steps, warmup)
    which = "BASELINE.json configs[4] shape: 4 x 8192 codes, e_dim 256" if CONFIG == "c5" else "BASELINE.json configs[2]"
    return {"workload": f"full index generation + collision resolution, {items} synthetic 4096-d items per GPU "
                        f"({which}; x{gpus} GPUs = configs[3] shape); the reference arm (--impl reference) runs the "
                        f"unmodified index/generate_indices.py on a bounded sample of {n_ref} items of the same stream per step "
                        f"(configs[0] is 25000)",
            "items_per_gpu": items, "reference_sample_items": n_ref, "in_dim": DIMS[0], "encoder": DIMS, "levels": len(N_CODES),
            "codes_per_level": N_CODES[0], "e_dim": E_DIM, "sk_epsilon_last": EPS_LAST, "sk_iters": SK_ITERS, "max_rounds": 20,
            "l2_policy": "inputs (16.4 GB/GPU) larger than L2, no flush", "parallelism": f"items sharded x{gpus}"}


# ----------------------------------------------------------------------------- GPU arm
DUMP_BYTES = 64 << 20        # --dump-outputs: bytes written in all (all ranks together)


def dump_outputs(out_dir, arrays, budget):
    """Each array as out_dir/<name>.npy, float64 arrays as float64 and everything else as float32 (codes < 2^24 are exact).
    Arrays larger than `budget` bytes in all keep a fixed, seeded sample of their rows (the same rows for the same
    shape in every run), written in ascending row order with the row numbers beside them as <name>_rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v.detach().cpu() if hasattr(v, "detach") else v) for k, v in arrays.items()}
    arrays = {k: v.astype(np.float64 if v.dtype == np.float64 else np.float32) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    with_rows = sum(v.nbytes + 8 * v.shape[0] for v in arrays.values() if v.ndim)
    for name, v in arrays.items():
        if total > budget and v.ndim and v.shape[0] > 1:
            keep = max(1, int(v.shape[0] * budget / with_rows))
            rows = np.sort(np.random.default_rng(SEED_X).choice(v.shape[0], keep, replace=False))
            v = v[rows]
            np.save(os.path.join(out_dir, f"{name}_rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(out_dir, f"{name}.npy"), v)


def run_gpu_arm(a):
    import torch
    import torch.distributed as dist
    from lcrec_b200 import ops
    from lcrec_b200.distributed import CudaBackend, ShardPlan, generate_codes_sharded
    from lcrec_b200.models import RQVAE

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    device = torch.device(f"cuda:{local}")
    torch.cuda.set_device(device)
    if world > 1:
        # NCCL prints its version banner / debug lines on stdout while the communicator is created: point fd 1
        # at stderr for that moment so that stdout carries nothing but the single JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=device)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    pk = peaks()
    ops.set_default_engine(a.engine)
    if os.environ.get("LCREC_SPECULATIVE") in ("0", "1", "2"):      # A/B of the late collision rounds: 0 host read per round, 1 blind, 2 graph replays (default)
        ops.indexer_set_speculative(int(os.environ["LCREC_SPECULATIVE"]))
    ws, bs, cbs, head = make_model()
    n_local = a.items
    model = RQVAE(in_dim=DIMS[0], num_emb_list=N_CODES, e_dim=E_DIM, layers=DIMS[1:-1], sk_epsilons=[0.0, 0.0, 0.0, EPS_LAST],
                  sk_iters=SK_ITERS)
    sd = model.state_dict()
    lin = sorted([k for k in sd if k.startswith("encoder.mlp_layers.") and k.endswith(".weight")], key=lambda s: int(s.split(".")[2]))
    for k, w, b in zip(lin, ws, bs):
        sd[k] = torch.from_numpy(w); sd[k.replace(".weight", ".bias")] = torch.from_numpy(b)
    for l, cb in enumerate(cbs):
        sd[f"rq.vq_layers.{l}.embedding.weight"] = torch.from_numpy(cb)
    model.load_state_dict(sd)
    model = model.to(device).eval()
    x = make_items_device(n_local, head, device, rank)
    plan = ShardPlan(n_local * world, world)
    backend = CudaBackend(model, n_local, a.chunk_rows)
    ix = backend.indexer

    def step():
        if world == 1:
            return ix.run_device(x, 20)
        return generate_codes_sharded(backend, x, plan, rank, 20)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(a.warmup):
        codes, stats = step()
    barrier()
    ops.profile_enable(True)
    ops.profile_collect()
    launches0 = ops.launch_count()
    sampler = ClockSampler(local) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if a.profile_window:
        torch.cuda.profiler.start()
    e0.record()
    for _ in range(a.steps):
        codes, stats = step()
    e1.record()
    barrier()
    if a.profile_window:
        torch.cuda.profiler.stop()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"codes" if world == 1 else f"codes_rank{rank}": codes}, DUMP_BYTES // world)
    launches = ops.launch_count() - launches0
    prof = ops.profile_collect()
    ops.profile_enable(False)
    t = torch.tensor([ms_total], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / a.steps
    value = n_local * world / (ms_step * 1e-3)

    # ---- end to end through the host-buffer C-ABI call (pinned input, H2D + D2H inside the timed region)
    e2e = None
    if not a.no_e2e:
        n_e2e = min(n_local, a.e2e_items)
        xh = torch.empty((n_e2e, DIMS[0]), dtype=torch.float32, pin_memory=True)
        xh.copy_(x[:n_e2e])
        out_h = torch.empty((n_e2e, len(N_CODES)), dtype=torch.int64, pin_memory=True)
        ix.run_host(xh, out_h, 20)
        barrier()
        t0 = time.perf_counter()
        e0.record()
        reps = max(1, min(a.steps, 3))
        for _ in range(reps):
            ix.run_host(xh, out_h, 20)
        e1.record()
        barrier()
        ms_e = e0.elapsed_time(e1) / reps
        te = torch.tensor([ms_e], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        # what the host link alone allows: the same pinned buffer copied to the device in the same chunks, no compute
        # (all ranks at once: at N = 8 the ranks share the host's memory system and PCIe root complexes)
        stage = torch.empty((min(a.chunk_rows, n_e2e), DIMS[0]), dtype=torch.float32, device=device)
        barrier()
        e0.record()
        for s0 in range(0, n_e2e, stage.shape[0]):
            m0 = min(stage.shape[0], n_e2e - s0)
            stage[:m0].copy_(xh[s0:s0 + m0], non_blocking=True)
        e1.record()
        barrier()
        tc = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(tc, op=dist.ReduceOp.MAX)
        h2d_gbs = n_e2e * DIMS[0] * 4 * world / (float(tc.item()) * 1e-3) / 1e9
        del stage
        e2e = {"value": n_e2e * world / (float(te.item()) * 1e-3), "unit": "items/s", "h2d_bytes_per_step": n_e2e * DIMS[0] * 4,
               "h2d_only_gbs_all_ranks": h2d_gbs, "h2d_only_items_per_s": h2d_gbs * 1e9 / (DIMS[0] * 4),
               "d2h_bytes_per_step": n_e2e * len(N_CODES) * 8, "items_per_gpu": n_e2e,
               "note": "lcrec_indexer_run_host: pinned host embeddings -> codes in host memory; each rank indexes its own items"}
        del xh

    # ---- multi-GPU correctness, untimed: the sharded path over a union of subsets == ONE GPU over the same union (bit for bit)
    sharded_ok = None
    if world > 1:
        n_sub = min(n_local, max(1024, a.check_items // world))
        sub_plan = ShardPlan(n_sub * world, world)
        c_sh, _ = generate_codes_sharded(backend, x[:n_sub], sub_plan, rank, 20)
        all_codes = torch.empty((n_sub * world, c_sh.shape[1]), dtype=c_sh.dtype, device=device)
        dist.all_gather_into_tensor(all_codes, c_sh.contiguous())
        all_x = torch.empty((n_sub * world, DIMS[0]), dtype=torch.float32, device=device) if rank == 0 else None
        dist.gather(x[:n_sub].contiguous(), list(all_x.split(n_sub)) if rank == 0 else None, dst=0)
        flag = torch.zeros(1, dtype=torch.int64, device=device)
        if rank == 0:
            c_one, _ = ix.run_device(all_x, 20)
            flag[0] = int(torch.equal(c_one, all_codes))
            del all_x
        dist.broadcast(flag, src=0)
        sharded_ok = {"equal": bool(flag.item()), "items": n_sub * world,
                      "note": "generate_codes_sharded over the ranks' first items vs lcrec_indexer_run_device on rank 0 over their union"}
    # ---- `.index.json` emission of this rank's table (generate_indices.py:138-145), outside the timed region like in the script
    json_ms = None
    if rank == 0:
        cdev = codes.to(device) if not codes.is_cuda else codes
        ops.index_json_bytes(cdev[:1024])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        blob = ops.index_json_bytes(cdev)
        json_ms = {"device_emitter_ms": (time.perf_counter() - t0) * 1e3, "bytes": len(blob), "rows": int(cdev.shape[0]),
                   "note": "lcrec_index_json + one D2H of the text; the reference's Python dict + json.dump is ~2 us/row"}
        del blob
    if rank == 0:
        # roofline of the dominant kernel: encoder layer 1 (4096 -> 2048)
        l1_ms, l1_calls = prof.get(1, (0.0, 0))
        rows_per_launch = min(a.chunk_rows, n_local)
        flops_launch = 2.0 * DIMS[0] * DIMS[1] * (n_local * a.steps / max(l1_calls, 1))
        ach = flops_launch / (l1_ms / max(l1_calls, 1) * 1e-3) / 1e12 if l1_calls else None
        stage_ms = {str(k): round(v[0] / a.steps, 4) for k, v in sorted(prof.items())}
        eng = ("f16 x3, linear_pair_kernel<64,3> (tcgen05 cta_group::2, 256x256 tiles, persistent)" if a.engine == 1
               else "tf32 x3, linear_split3_kernel<256,16,4,false>")
        traffic = None
        traffic_src = None
        for name in ("r2_pair_ncu_summary.json", "r1_v5_pair_ncu_summary.json"):
            try:   # DRAM bytes of one launch of this kernel from the committed ncu --set full capture (same rows per launch)
                summ = json.load(open(os.path.join(ROOT, "profiles", name)))["layer1"]
                if a.engine == 1 and summ["rows_per_launch"] == rows_per_launch and CONFIG == "c3":
                    traffic = summ["dram_bytes_read"] + summ["dram_bytes_write"]
                    traffic_src = name
                    break
            except Exception:  # noqa: BLE001
                traffic = None
        roof = {"bound": "tensor", "kernel": f"{eng} (encoder layer 1, 4096->2048)",
                "achieved": ach, "peak": pk["bf16_sustained"], "unit": "TFLOP/s", "frac": (ach / pk["bf16_sustained"]) if ach else None,
                "traffic": traffic, "traffic_unit": f"bytes of DRAM read + write per launch (ncu --set full, profiles/{traffic_src}); "
                                                    "algorithmic: 2.18 GB operands + 1.07 GB output",
                "peak_source": pk["source"] + ", bf16 dense sustained",
                "note": "achieved = algorithmic fp32 GEMM FLOPs (2*M*4096*2048 per launch) / CUDA-event launch time; the kernel issues 3 MMAs "
                        "per product (fp32-accurate two-term operand split): tensor work = 3x achieved; ceiling = peak/3 with f16 operands "
                        "(kind::f16 runs at the bf16 rate), peak/6 with tf32 operands.  ncu: tensor pipe 91 % active at the power-capped clock",
                "tensor_work_tflops": 3 * ach if ach else None,
                "frac_of_split_ceiling": (ach / (pk["bf16_sustained"] / (3 if a.engine == 1 else 6))) if ach else None,
                "launches": l1_calls, "avg_launch_ms": l1_ms / max(l1_calls, 1), "rows_per_launch": rows_per_launch,
                "kernel_share_of_step": l1_ms / a.steps / ms_step,
                "hbm_frac_end_to_end": value / world * BYTES_PER_ITEM / 1e9 / pk["hbm_gbs"], "stage_ms_per_step": stage_ms}
        # second roofline: the per-group Sinkhorn of round 1 against the MEASURED fp64 FMA peak.  Algorithmic fp64 work = 2 K FMAs per row
        # per iteration (SURVEY 8(d): 25 600 FMAs per row at K = 256, 50 iterations); reciprocals, exp and the literal last step excluded
        sk = None
        try:
            peak64 = ops.fp64_peak_tflops(device)
            ms22 = prof.get(22, (0.0, 0))[0] / a.steps
            rows1 = stats["rows_round1"] / (world if world > 1 else 1)
            ach64 = 2.0 * rows1 * 2 * N_CODES[-1] * SK_ITERS / (ms22 * 1e-3) / 1e12 if ms22 > 0 else None
            sk = {"bound": "fp64", "kernel": "per-group Sinkhorn, first round (stage 22)", "achieved": ach64, "peak": peak64, "unit": "TFLOP/s",
                  "frac": (ach64 / peak64) if ach64 else None, "rows_per_rank": rows1, "ms": ms22,
                  "peak_source": "measured in this run (lcrec_fp64_peak_probe: 8 independent DFMA chains per thread)",
                  "note": "algorithmic = 2 K FMAs per row per iteration; per iteration a group also needs K + n reciprocals (~5 fp64 ops each: as "
                          "much work as the FMAs at n = 2), so the pipe is busier than this fraction says"}
        except Exception as exc:  # noqa: BLE001
            sk = {"error": str(exc)}
        cpu = None
        torch_cuda = None
        if world == 1 and not a.no_cpu:
            cpu, _ = cpu_baseline(ws, bs, cbs, a.cpu_sample or C1_ITEMS)
            if not a.no_torch_cuda:
                # the reference on its own GPU path (torch-CUDA / cuBLAS fp32), same script, same items: the honest GPU comparator
                res = run_reference_script(ws, bs, cbs, reference_items(a.cpu_sample or C1_ITEMS), f"cuda:{local}", 2, host_cores(), 600)
                if "unavailable" in res:
                    torch_cuda = res
                else:
                    torch_cuda = {"value": res["items"] / res["seconds"][-1], "unit": "items/s", "items": res["items"], "seconds": res["seconds"][-1],
                                  "rounds": res["rounds"], "note": "unmodified index/generate_indices.py with device=cuda:0 (second of two runs)"}
        line = {"metric": "items indexed/sec (4-level RQ + Sinkhorn collision resolution)", "value": value, "unit": "items/s",
                "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic (low-rank parents + noise, random-init encoder, k-means-style codebooks)",
                "config": workload_config(world, n_local, a.steps, a.warmup, a.cpu_sample), "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
                "roofline": roof, "roofline_sinkhorn": sk, "cpu_baseline": cpu, "reference_torch_cuda": torch_cuda, "index_json": json_ms, "sharded_equals_single": sharded_ok, "stats": stats,
                "flop_per_item": FLOP_PER_ITEM, "bytes_per_item": BYTES_PER_ITEM,
                "algorithmic_tflops_end_to_end": value * FLOP_PER_ITEM / 1e12}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


# ----------------------------------------------------------------------------- c2: the training epoch (BASELINE configs[1])
C2_ITEMS, C2_BATCH = 25_000, 1024
C2_FLOP_PER_ITEM = 3 * 2 * 2 * sum(a * b for a, b in zip(DIMS[:-1], DIMS[1:])) + 4 * 2 * 256 * 32      # fwd + dgrad + wgrad, encoder + decoder


def c2_reference_batches(steps, warmup):
    return int(min(25, max(2, 100 // max(steps + warmup, 1))))


def c2_weights():
    from lcrec_b200.synth import seeded_weights
    ws, bs, cbs = seeded_weights(DIMS, N_CODES, E_DIM, seed=SEED_W, cb_scale=0.3)
    wd, bd, _ = seeded_weights(DIMS[::-1], N_CODES, E_DIM, seed=SEED_W + 1)
    return ws, bs, wd, bd, cbs


def c2_config(gpus, steps, warmup, bn):
    nb = c2_reference_batches(steps, warmup)
    return {"workload": f"RQ-VAE training epoch (BASELINE.json configs[1], index/main.py + run.sh shape): {C2_ITEMS} synthetic 4096-d items, "
                        f"batch {C2_BATCH} (24 full batches + one of 424), AdamW lr 1e-3 wd 1e-4, linear warm-up, clip 1.0, Sinkhorn "
                        f"(eps 0.003, 50 it) on level 4, bn={bn}; a step = one epoch; the reference arm times the unmodified "
                        f"Trainer._train_epoch on {nb} batches per step",
            "items": C2_ITEMS, "batch": C2_BATCH, "bn": bn, "encoder": DIMS, "levels": 4, "codes_per_level": 256, "e_dim": E_DIM,
            "reference_sample_batches": nb, "l2_policy": "22 M parameters + Adam state (358 MB) and the batch stream exceed L2; no flush",
            "parallelism": f"data parallel x{gpus}" if gpus > 1 else "single GPU"}


def run_reference_train(ws, bs, wd, bd, cbs, x, device, repeat, threads, bn, timeout_s=1500):
    runner = os.path.join(ROOT, "baseline", "run_reference_train.py")
    if not os.path.isfile(os.path.join(ROOT, "baseline", "_ref", "index", "trainer.py")):
        return {"unavailable": "baseline/_ref/index not staged"}
    tmp = tempfile.mkdtemp(prefix="lcrec_reftrain_")
    npz, out = os.path.join(tmp, "in.npz"), os.path.join(tmp, "out.json")
    arrs = {"x": x}
    for i, (w, b, w2, b2) in enumerate(zip(ws, bs, wd, bd)):
        arrs[f"w{i}"] = w; arrs[f"b{i}"] = b; arrs[f"wd{i}"] = w2; arrs[f"bd{i}"] = b2
    for l, cb in enumerate(cbs):
        arrs[f"cb{l}"] = cb
    np.savez(npz, **arrs)
    env = dict(os.environ)
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
        env[k] = str(threads)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "PYTHONPATH"):
        env.pop(k, None)
    try:
        r = subprocess.run([sys.executable, runner, "--npz", npz, "--device", device, "--threads", str(threads), "--repeat", str(repeat),
                            "--bn", str(int(bn)), "--out", out], env=env, cwd=tmp, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                           timeout=timeout_s)
        if r.returncode != 0 or not os.path.exists(out):
            return {"unavailable": f"runner exit {r.returncode}: {r.stderr.strip()[-300:]}"}
        return json.load(open(out))
    except subprocess.TimeoutExpired:
        return {"unavailable": f"runner exceeded {timeout_s} s"}


def c2_cpu_baseline(n_batches, repeat, drop, bn):
    ws, bs, wd, bd, cbs = c2_weights()
    x = reference_items(n_batches * C2_BATCH)
    res = run_reference_train(ws, bs, wd, bd, cbs, x, "cpu", repeat, host_cores(), bn)
    if "unavailable" in res:
        return {"value": None, "unit": "items/s", "cores": host_cores(), "kind": "reference", "sample": res["unavailable"]}, None
    secs = res["seconds"][drop:]
    dt = float(np.mean(secs))
    return {"value": res["items"] / dt, "unit": "items/s", "cores": int(res["torch_threads"]), "kind": "reference", "seconds": dt,
            "host_cpus": res["cpu_count"], "torch": res["torch"],
            "sample": f"{n_batches} batches of {C2_BATCH} ({res['items']} items) per run: the UNMODIFIED Trainer._train_epoch "
                      f"(baseline/_ref/index/trainer.py:98-125, torch CPU), {len(secs)} timed run(s)"}, dt


def run_c2_reference(a):
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    nb = c2_reference_batches(a.steps, a.warmup)
    cpu, dt = c2_cpu_baseline(nb, a.warmup + a.steps, a.warmup, a.bn)
    line = {"impl": "reference", "metric": "items trained/sec (RQ-VAE training epoch, batch 1024)", "value": cpu["value"], "unit": "items/s",
            "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": None if dt is None else dt * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": c2_config(a.gpus, a.steps, a.warmup, a.bn),
            "cpu_baseline": cpu, "e2e": {"value": cpu["value"], "unit": "items/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)
    return 0


def run_c2(a):
    """One step = one training epoch through lcrec_b200.trainer.Trainer._train_epoch (the reference's loop, trainer.py:98-125)."""
    import torch
    from lcrec_b200 import ops
    from lcrec_b200.models import RQVAE
    import lcrec_b200.trainer as TR
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        raise SystemExit("bench.py --config c2 measures the single-GPU epoch; the data-parallel trainer is scripts/check_dp_trainer.py")
    device = torch.device("cuda:0")
    torch.cuda.set_device(device)
    pk = peaks()
    ws, bs, wd, bd, cbs = c2_weights()

    def build(bn):
        m = RQVAE(in_dim=DIMS[0], num_emb_list=N_CODES, e_dim=E_DIM, layers=DIMS[1:-1], bn=bn, kmeans_init=False,
                  sk_epsilons=[0.0, 0.0, 0.0, EPS_LAST], sk_iters=SK_ITERS)
        sd = m.state_dict()
        stride = 4 if bn else 3
        for i, (w, b, w2, b2) in enumerate(zip(ws, bs, wd, bd)):
            sd[f"encoder.mlp_layers.{1 + stride * i}.weight"] = torch.from_numpy(w); sd[f"encoder.mlp_layers.{1 + stride * i}.bias"] = torch.from_numpy(b)
            sd[f"decoder.mlp_layers.{1 + stride * i}.weight"] = torch.from_numpy(w2); sd[f"decoder.mlp_layers.{1 + stride * i}.bias"] = torch.from_numpy(b2)
        for l, cb in enumerate(cbs):
            sd[f"rq.vq_layers.{l}.embedding.weight"] = torch.from_numpy(cb)
        m.load_state_dict(sd)
        args = argparse.Namespace(lr=1e-3, epochs=10000, batch_size=C2_BATCH, num_workers=0, eval_step=50, learner="AdamW",
                                  lr_scheduler_type="linear", warmup_epochs=50, data_path="", weight_decay=1e-4, dropout_prob=0.0, bn=bn,
                                  loss_type="mse", kmeans_init=False, kmeans_iters=100, sk_epsilons=[0.0, 0.0, 0.0, EPS_LAST], sk_iters=SK_ITERS,
                                  device="cuda:0", num_emb_list=N_CODES, e_dim=E_DIM, quant_loss_weight=1.0, beta=0.25, layers=DIMS[1:-1],
                                  save_limit=5, ckpt_dir=tempfile.mkdtemp(prefix="lcrec_c2_"))
        return TR.Trainer(args, m, 25)

    import logging
    logging.disable(logging.CRITICAL)
    xh = torch.from_numpy(reference_items(C2_ITEMS)).pin_memory()
    host_loader = [xh[s:s + C2_BATCH] for s in range(0, C2_ITEMS, C2_BATCH)]
    xd = xh.to(device)
    dev_loader = [xd[s:s + C2_BATCH] for s in range(0, C2_ITEMS, C2_BATCH)]
    os.environ.setdefault("TQDM_DISABLE", "1")

    def timed(tr, loader, steps, warmup):
        with open(os.devnull, "w") as devnull, contextlib_redirect(devnull):
            for ep in range(warmup):
                tr._train_epoch(loader, ep)
            torch.cuda.synchronize()
            n0 = ops.launch_count() + (tr._gstep.replayed_launches if getattr(tr, "_gstep", None) is not None else 0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for ep in range(steps):
                losses = tr._train_epoch(loader, warmup + ep)
            e1.record()
            torch.cuda.synchronize()
        n1 = ops.launch_count() + (tr._gstep.replayed_launches if getattr(tr, "_gstep", None) is not None else 0)
        return e0.elapsed_time(e1) / steps, n1 - n0, losses

    tr = build(a.bn)
    # untimed: the step of every batch size runs eagerly 3 times and is then captured; the batch of 424 occurs once per epoch,
    # so its graph exists from the 5th epoch on (a capture inside the timed region would cost ~0.2 s)
    for ep in range(5):
        with open(os.devnull, "w") as devnull, contextlib_redirect(devnull):
            tr._train_epoch(dev_loader, ep)
    sampler = ClockSampler(0)
    ms_step, launches, losses = timed(tr, dev_loader, a.steps, a.warmup)
    clocks = sampler.stop()
    ms_e2e, _, _ = timed(tr, host_loader, max(1, min(a.steps, 3)), 1)
    g = tr._gstep
    extra = {}
    if not a.no_cpu:
        other = build(not a.bn)
        ms_other, _, _ = timed(other, dev_loader, 2, 5)
        extra["bn_" + str(not a.bn).lower() + "_ms_per_step"] = ms_other
        del other
        monkey = TR.TRAIN_GRAPH
        TR.TRAIN_GRAPH = False
        eager = build(a.bn)
        ms_eager, _, _ = timed(eager, dev_loader, 2, 1)
        TR.TRAIN_GRAPH = monkey
        extra["eager_launches_ms_per_step"] = ms_eager
        del eager
    value = C2_ITEMS / (ms_step * 1e-3)
    ach = value * C2_FLOP_PER_ITEM / 1e12
    cpu = None
    if not a.no_cpu:
        cpu, _ = c2_cpu_baseline(12, 1, 0, a.bn)
    line = {"metric": "items trained/sec (RQ-VAE training epoch, batch 1024)", "value": value, "unit": "items/s", "n_gpus": 1, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms_step, "ms_per_batch": ms_step / len(dev_loader), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic (low-rank parents + noise, seeded weights)",
            "config": c2_config(1, a.steps, a.warmup, a.bn), "clocks": clocks,
            "e2e": {"value": C2_ITEMS / (ms_e2e * 1e-3), "unit": "items/s", "h2d_bytes_per_step": C2_ITEMS * DIMS[0] * 4, "d2h_bytes_per_step": 25 * 32,
                    "note": "Trainer._train_epoch over pinned host batches: H2D of every batch and the per-step loss read-back inside the timed region"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": "whole training step (encoder + decoder GEMMs forward, dgrad, wgrad; 3 MMAs per fp32 product)",
                         "achieved": ach, "peak": pk["bf16_sustained"], "unit": "TFLOP/s", "frac": ach / pk["bf16_sustained"], "traffic": None,
                         "peak_source": pk["source"] + ", bf16 dense sustained",
                         "note": "algorithmic FLOPs 134.3 MFLOP/item (SURVEY 8(d)) / epoch time; ceiling = peak / 3 (fp32-accurate operand split); "
                                 "at batch 1024 the GEMMs fill 32 of 74 CTA-pair tiles, so the step is latency / occupancy bound, not pipe bound"},
            "cpu_baseline": cpu, "losses_last_epoch": [float(v) for v in losses],
            "cuda_graph": None if g is None else {"replays": g.replays, "eager_steps": g.eager_steps, "capture_error": g.capture_error},
            **extra}
    print(json.dumps(line), flush=True)
    return 0


class contextlib_redirect:
    """stderr -> a sink (tqdm bars of the trainer), stdout untouched."""
    def __init__(self, sink):
        self.sink = sink

    def __enter__(self):
        self.old = sys.stderr
        sys.stderr = self.sink

    def __exit__(self, *exc):
        sys.stderr = self.old
        return False


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--items", type=int, default=1_000_000, help="items per GPU")
    ap.add_argument("--chunk-rows", dest="chunk_rows", type=int, default=131072)
    ap.add_argument("--e2e-items", dest="e2e_items", type=int, default=1_000_000)
    ap.add_argument("--cpu-sample", dest="cpu_sample", type=int, default=None,
                    help="items per run of the unmodified reference script: default 25000 (C1) for the cpu_baseline leg of the GPU arm, "
                         "reference_sample_items(steps, warmup) per step for --impl reference")
    ap.add_argument("--engine", type=int, default=1, choices=[0, 1], help="GEMM operand encoding: 1 = f16 x3 (default), 0 = tf32 x3")
    ap.add_argument("--check-items", dest="check_items", type=int, default=200_000,
                    help="N > 1: items of the untimed sharded-vs-single-GPU equality check (over all ranks)")
    ap.add_argument("--no-e2e", dest="no_e2e", action="store_true")
    ap.add_argument("--no-cpu", dest="no_cpu", action="store_true")
    ap.add_argument("--no-torch-cuda", dest="no_torch_cuda", action="store_true", help="skip the reference-on-torch-CUDA comparator")
    ap.add_argument("--profile-window", dest="profile_window", action="store_true",
                    help="cudaProfilerStart/Stop around the timed steps (for ncu --profile-from-start off)")
    ap.add_argument("--config", default="c3", choices=["c3", "c2", "c5"],
                    help="c3: index generation, 4 x 256 codes (default; BASELINE configs[2] / [3]); c5: 4 x 8192 codes, e_dim 256 "
                         "(configs[4]; --items defaults to 100000); c2: the training epoch (configs[1])")
    ap.add_argument("--bn", action="store_true", help="c2: BatchNorm in the encoder / decoder (what `run.sh --bn False` really trains)")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="c3 / c5: write the codes of the last timed step as DIR/codes.npy (float32; DIR/codes_rank<r>.npy per rank "
                         "for N > 1), at most 64 MB in all: larger tables keep a fixed, seeded sample of rows (DIR/<name>_rows.npy)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl == "reference" or a.config == "c2"):
        ap.error("--dump-outputs applies to the GPU arm of --config c3 / c5")
    a.warmup = max(a.warmup, 0)
    set_config(a.config)
    if a.config == "c5":
        if a.items == 1_000_000:
            a.items = 100_000
        a.e2e_items = min(a.e2e_items, a.items)
        a.cpu_sample = a.cpu_sample or 4096       # the reference's per-group Sinkhorn over 8192 columns is ~40x the c3 cost per row
    if a.config == "c2":
        return run_c2_reference(a) if a.impl == "reference" else run_c2(a)
    if a.impl == "reference":
        return run_reference_arm(a)
    return run_gpu_arm(a)


if __name__ == "__main__":
    sys.exit(main())
