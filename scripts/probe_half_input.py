"""Half-precision embedding input on one GPU, in one run (writes one JSON, default profiles/r3_half_input.json):

  device   1 M items (the c3 model and items of bench.py), ms per Indexer.run_device pass for fp32 / bf16 / fp16, the dtypes
           interleaved after a warm-up of each, CUDA events; then, in a separate profiled pass, the input-split stage
           (profile tag 0) and layer 1 (tag 1) per dtype;
  host     1 M items in pinned host memory, Indexer.run_host items/s for fp32 and fp16, next to the H2D-only ceiling of the same
           bytes (the pinned buffer copied to the device in the same chunks, no compute - as bench.py measures it);
  10 M     10 M bf16 items device-resident on this one GPU (the 1 M-item streams of ranks 0..9 of bench.py's weak scaling,
           configs[3] at full size): ms per pass, items/s, memory, generation stats - fp32 (164 GB) does not fit;
  equal    codes of bf16 / fp16 input against the fp32 path on the upcast input (device and host input; must be 0 rows), and,
           as information, the rows whose codes change because the input was rounded to bf16 / fp16, with collision rates;
  card     name, power limit and clocks (nvidia-smi, query only) in the same run.

    python scripts/probe_half_input.py [--items 1000000] [--big-items 10000000] [--steps 5] [--out PATH]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
from lcrec_b200 import ops  # noqa: E402
from lcrec_b200 import generate_indices as G  # noqa: E402
from lcrec_b200.models import RQVAE  # noqa: E402

DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}


def card(dev_index: int) -> dict:
    q = "name,power.limit,power.max_limit,clocks.sm,clocks.max.sm,clocks.mem,temperature.gpu"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", str(dev_index)],
                       capture_output=True, text=True)
    vals = [v.strip() for v in r.stdout.strip().split(",")]
    return dict(zip(q.split(","), vals)) if r.returncode == 0 and len(vals) == len(q.split(",")) else {"error": r.stderr.strip()}


def build_model(dev):
    ws, bs, cbs, head = bench.make_model()
    model = RQVAE(in_dim=bench.DIMS[0], num_emb_list=bench.N_CODES, e_dim=bench.E_DIM, layers=bench.DIMS[1:-1],
                  sk_epsilons=[0.0, 0.0, 0.0, bench.EPS_LAST], sk_iters=bench.SK_ITERS)
    sd = model.state_dict()
    lin = sorted([k for k in sd if k.startswith("encoder.mlp_layers.") and k.endswith(".weight")], key=lambda s: int(s.split(".")[2]))
    for k, w, b in zip(lin, ws, bs):
        sd[k] = torch.from_numpy(w); sd[k.replace(".weight", ".bias")] = torch.from_numpy(b)
    for l, cb in enumerate(cbs):
        sd[f"rq.vq_layers.{l}.embedding.weight"] = torch.from_numpy(cb)
    model.load_state_dict(sd)
    return model.to(dev).eval(), head


def timed(fn, e0, e1):
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def rows_differing(a, b) -> int:
    return int((a != b).any(dim=1).sum().item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--items", type=int, default=1_000_000)
    ap.add_argument("--big-items", type=int, default=10_000_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--chunk-rows", type=int, default=131072)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_half_input.json"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "probe_half_input needs a B200"
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    res = {"card_before": card(0), "torch": torch.__version__, "cuda": torch.version.cuda, "items": a.items,
           "chunk_rows": a.chunk_rows, "steps": a.steps}
    model, head = build_model(dev)
    n = a.items
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    # ---------------------------------------------------------------- device-resident, 1 M items
    x = {"fp32": bench.make_items_device(n, head, dev, 0)}
    x["bf16"] = x["fp32"].to(torch.bfloat16)
    x["fp16"] = x["fp32"].to(torch.float16)
    ix = G.build_indexer(model, n, a.chunk_rows)
    out = {}
    for name in DTYPES:                                      # warm-up of every shape
        out[name] = ix.run_device(x[name], 20)
    ms = {name: [] for name in DTYPES}
    for _ in range(a.steps):                                 # interleaved
        for name in DTYPES:
            t, out[name] = timed(lambda: ix.run_device(x[name], 20), e0, e1)
            ms[name].append(t)
    ops.profile_enable(True)
    ops.profile_collect()
    stages = {}
    for name in DTYPES:
        for _ in range(2):
            ix.run_device(x[name], 20)
        prof = ops.profile_collect()
        stages[name] = {"input_split_ms_per_pass": prof.get(0, (0.0, 0))[0] / 2, "input_split_calls_per_pass": prof.get(0, (0, 0))[1] / 2,
                        "layer1_ms_per_pass": prof.get(1, (0.0, 0))[0] / 2}
    ops.profile_enable(False)
    dev_res = {}
    for name in DTYPES:
        s = sorted(ms[name])
        dev_res[name] = {"ms_per_pass": s, "ms_median": s[len(s) // 2], "items_per_s_median": n / (s[len(s) // 2] * 1e-3),
                         "input_bytes_per_item": bench.DIMS[0] * x[name].element_size(), **stages[name],
                         "collision_rate": (n - out[name][1]["n_unique"]) / n, "stats": out[name][1]}
    res["device_1m"] = dev_res

    # equality: half input == fp32 path on the upcast input
    eq = {}
    for name in ("bf16", "fp16"):
        up = x[name].to(torch.float32)
        c_up, s_up = ix.run_device(up, 20)
        del up
        eq[name] = {"rows_differing_from_fp32_upcast_device": rows_differing(out[name][0], c_up), "stats_equal_device": s_up == out[name][1],
                    "rows_changed_by_rounding_the_input": rows_differing(out[name][0], out["fp32"][0]),
                    "collision_rate_fp32_input": dev_res["fp32"]["collision_rate"], "collision_rate": dev_res[name]["collision_rate"]}
        eq[name]["_codes_up"] = c_up.cpu()

    # ---------------------------------------------------------------- host-resident, 1 M items, pinned
    host = {}
    xh = {}
    for name in ("fp32", "fp16"):
        xh[name] = torch.empty((n, bench.DIMS[0]), dtype=DTYPES[name], pin_memory=True)
        xh[name].copy_(x[name])
    out_h = torch.empty((n, len(bench.N_CODES)), dtype=torch.int64, pin_memory=True)
    codes_h = {}
    for name in xh:                                          # warm-up
        ix.run_host(xh[name], out_h, 20)
    t_host = {name: [] for name in xh}
    for _ in range(3):
        for name in xh:
            torch.cuda.synchronize()
            t, r = timed(lambda: ix.run_host(xh[name], out_h, 20), e0, e1)
            t_host[name].append(t)
            codes_h[name] = (out_h.clone(), r[1])
    for name in xh:
        stage = torch.empty((min(a.chunk_rows, n), bench.DIMS[0]), dtype=DTYPES[name], device=dev)
        torch.cuda.synchronize()
        e0.record()
        for s0 in range(0, n, stage.shape[0]):
            m0 = min(stage.shape[0], n - s0)
            stage[:m0].copy_(xh[name][s0:s0 + m0], non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        tc = e0.elapsed_time(e1)
        del stage
        nbytes = n * bench.DIMS[0] * xh[name].element_size()
        s = sorted(t_host[name])
        host[name] = {"ms_per_run": s, "items_per_s_median": n / (s[len(s) // 2] * 1e-3), "h2d_bytes": nbytes,
                      "h2d_only_ms": tc, "h2d_only_gbs": nbytes / (tc * 1e-3) / 1e9, "h2d_only_items_per_s": n / (tc * 1e-3)}
    res["host_1m_pinned"] = host
    eq["fp16"]["rows_differing_from_fp32_upcast_host"] = rows_differing(codes_h["fp16"][0], eq["fp16"]["_codes_up"])
    eq["fp16"]["stats_equal_host"] = codes_h["fp16"][1] == out["fp16"][1]
    eq["fp32_host_vs_device_rows_differing"] = rows_differing(codes_h["fp32"][0], out["fp32"][0].cpu())
    for name in ("bf16", "fp16"):
        del eq[name]["_codes_up"]
    res["equality_1m"] = eq
    del xh, out_h, x, out, ix
    torch.cuda.synchronize()
    torch.cuda.empty_cache()

    # ---------------------------------------------------------------- 10 M bf16 items on one GPU
    if a.big_items > 0:
        nb = a.big_items
        per = n
        xb = torch.empty((nb, bench.DIMS[0]), dtype=torch.bfloat16, device=dev)
        for p in range((nb + per - 1) // per):
            m0 = min(per, nb - p * per)
            xb[p * per: p * per + m0].copy_(bench.make_items_device(m0, head, dev, p))
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        ix = G.build_indexer(model, nb, a.chunk_rows)
        torch.cuda.reset_peak_memory_stats(dev)
        c, st = ix.run_device(xb, 20)                         # warm-up
        t_big = []
        for _ in range(2):
            t, (c, st) = timed(lambda: ix.run_device(xb, 20), e0, e1)
            t_big.append(t)
        free, total = torch.cuda.mem_get_info(dev)
        res["device_10m_bf16"] = {"items": nb, "ms_per_pass": t_big, "items_per_s": nb / (min(t_big) * 1e-3),
                                  "input_gb": xb.numel() * 2 / 1e9, "torch_peak_allocated_gb": torch.cuda.max_memory_allocated(dev) / 1e9,
                                  "device_used_gb_after": (total - free) / 1e9, "device_total_gb": total / 1e9,
                                  "stats": st, "collision_rate": (nb - st["n_unique"]) / nb,
                                  "note": "items = the 1 M-item streams of ranks 0..9 of bench.py (rank p: make_items_device(1 M, rank=p)), "
                                          "rounded to bf16; device_used includes the indexer's own workspace and torch's cache"}
        del xb, ix, c
    res["card_after"] = card(0)
    res["when"] = time.strftime("%Y-%m-%d %H:%M:%S")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in res if k in ("equality_1m", "card_before")}))
    print(json.dumps({name: {k: v for k, v in d.items() if k != "ms_per_pass"} for name, d in res["device_1m"].items()}))
    print(json.dumps(res["host_1m_pinned"]))
    print(json.dumps(res.get("device_10m_bf16")))


if __name__ == "__main__":
    main()
