"""torchrun --nproc-per-node N scripts/check_sharded_equals_single.py [n_total [dtype]] : item-sharded generation over N GPUs
(all-to-all bucket exchange, native rounds per owner) must reproduce the single-GPU table bit for bit.  dtype (float32 by
default, or float16 / bfloat16): the element type of the embeddings both runs read.  Prints one JSON line."""
import json, os, sys
import torch, torch.distributed as dist
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from lcrec_b200.distributed import CudaBackend, ShardPlan, generate_codes_sharded
from lcrec_b200.models import RQVAE
from lcrec_b200 import generate_indices as G

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
dev = torch.device(f"cuda:{local}")
torch.cuda.set_device(dev)
saved = os.dup(1); os.dup2(2, 1)
dist.init_process_group("nccl", device_id=dev)
dist.barrier(); torch.cuda.synchronize()
os.dup2(saved, 1); os.close(saved)
n_total = int(sys.argv[1]) if len(sys.argv) > 1 else 200_003          # odd: ragged shards
dtype = getattr(torch, sys.argv[2]) if len(sys.argv) > 2 else torch.float32
ws, bs, cbs, head = bench.make_model()
model = RQVAE(in_dim=4096, num_emb_list=bench.N_CODES, e_dim=32, layers=bench.DIMS[1:-1], sk_epsilons=[0.0, 0.0, 0.0, 0.003], sk_iters=50)
sd = model.state_dict()
lin = sorted([k for k in sd if k.startswith("encoder.mlp_layers.") and k.endswith(".weight")], key=lambda s: int(s.split(".")[2]))
for k, w, b in zip(lin, ws, bs):
    sd[k] = torch.from_numpy(w); sd[k.replace(".weight", ".bias")] = torch.from_numpy(b)
for l, cb in enumerate(cbs):
    sd[f"rq.vq_layers.{l}.embedding.weight"] = torch.from_numpy(cb)
model.load_state_dict(sd); model = model.to(dev).eval()
x_all = bench.make_items_device(n_total, head, dev, 0).to(dtype)        # the same items on every rank (rank argument fixed)
plan = ShardPlan(n_total, world)
backend = CudaBackend(model, plan.max_count)
codes_local, stats = generate_codes_sharded(backend, x_all[plan.slice(rank)].contiguous(), plan, rank, 20)
ref, ref_stats = G.generate_codes(model, x_all)                          # single-GPU run of the whole set on this rank
same = bool(torch.equal(codes_local.cpu(), ref[plan.slice(rank)]))
flag = torch.tensor([0 if same else 1], device=dev)
dist.all_reduce(flag)
ok = int(flag.item()) == 0 and stats["n_unique"] == ref_stats["n_unique"] and stats["rounds"] == ref_stats["rounds"]
if rank == 0:
    print(json.dumps({"world": world, "n_total": n_total, "dtype": str(dtype).replace("torch.", ""), "identical": int(flag.item()) == 0, "n_unique": stats["n_unique"],
                      "n_unique_single": ref_stats["n_unique"], "rounds": stats["rounds"], "ok": ok}), flush=True)
dist.barrier(); dist.destroy_process_group()
sys.exit(0 if ok else 1)
