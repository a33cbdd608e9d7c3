"""Training CLI with the flags of reference ``index/main.py`` (:14-94), including its
``type=bool`` quirk for --bn / --kmeans_init (any non-empty string, e.g. ``--bn False``, is True)."""
import argparse
import logging
import os
import random

import numpy as np
import torch
from torch.utils.data import DataLoader

from .datasets import EmbDataset
from .models.rqvae import RQVAE
from .trainer import Trainer


# flag, type, default - the command line of index/main.py:15-47; ``bool`` keeps the reference's quirk (any non-empty string,
# "False" included, parses to True); list defaults mean nargs="+"
FLAGS = [
    ("lr", float, 1e-3), ("epochs", int, 5000), ("batch_size", int, 2048), ("num_workers", int, 4), ("eval_step", int, 50),
    ("learner", str, "AdamW"), ("lr_scheduler_type", str, "constant"), ("warmup_epochs", int, 50),
    ("data_path", str, "../data/Games/Games.emb-llama-td.npy"), ("weight_decay", float, 0.0), ("dropout_prob", float, 0.0),
    ("bn", bool, False), ("loss_type", str, "mse"), ("kmeans_init", bool, True), ("kmeans_iters", int, 100),
    ("sk_epsilons", float, [0.0, 0.0, 0.0]), ("sk_iters", int, 50), ("device", str, "cuda:0"),
    ("num_emb_list", int, [256, 256, 256]), ("e_dim", int, 32), ("quant_loss_weight", float, 1.0), ("beta", float, 0.25),
    ("layers", int, [2048, 1024, 512, 256, 128, 64]), ("save_limit", int, 5), ("ckpt_dir", str, ""),
]


def build_parser(description="Index"):
    p = argparse.ArgumentParser(description=description)
    for name, kind, default in FLAGS:
        if isinstance(default, list):
            p.add_argument("--" + name, type=kind, nargs="+", default=default)
        else:
            p.add_argument("--" + name, type=kind, default=default)
    return p


def parse_args(argv=None):
    return build_parser().parse_args(argv)


def make_trainer(args, model, data_num, trainer_cls, dp_trainer_cls):
    """``trainer_cls`` on one device, or under torchrun (WORLD_SIZE > 1) ``dp_trainer_cls``: one process per GPU, every rank
    reads the same batches and trains its row block of each."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world <= 1:
        return trainer_cls(args, model, data_num)
    import torch.distributed as dist
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    args.device = f"cuda:{local_rank}"
    dist.init_process_group("nccl")
    return dp_trainer_cls(args, model, data_num)


def main(argv=None):
    seed = 2024
    random.seed(seed); np.random.seed(seed); torch.manual_seed(seed); torch.cuda.manual_seed_all(seed)
    args = parse_args(argv)
    print("=================================================")
    print(args)
    print("=================================================")
    logging.basicConfig(level=logging.DEBUG)
    data = EmbDataset(args.data_path)
    model = RQVAE(in_dim=data.dim, num_emb_list=args.num_emb_list, e_dim=args.e_dim, layers=args.layers,
                  dropout_prob=args.dropout_prob, bn=args.bn, loss_type=args.loss_type,
                  quant_loss_weight=args.quant_loss_weight, beta=args.beta, kmeans_init=args.kmeans_init,
                  kmeans_iters=args.kmeans_iters, sk_epsilons=args.sk_epsilons, sk_iters=args.sk_iters)
    print(model)
    loader = DataLoader(data, num_workers=args.num_workers, batch_size=args.batch_size, shuffle=True, pin_memory=True)
    from .dp_trainer import DataParallelTrainer
    best_loss, best_collision_rate = make_trainer(args, model, len(loader), Trainer, DataParallelTrainer).fit(loader)
    print("Best Loss", best_loss)
    print("Best Collision Rate", best_collision_rate)


if __name__ == "__main__":
    main()
