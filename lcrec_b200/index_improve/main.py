"""Training CLI of the EMA variant: the flags of reference ``index_improve/main.py`` (:15-125) - those of ``index/main.py``
plus --ema_decay / --epsilon / --reset_threshold / --reset_interval; ``--sk_epsilons`` defaults to zeros of the right
length (:87-89).  The reference's default device ``npu:0`` becomes ``cuda:0`` (this library is sm_100a only).  Under
torchrun (WORLD_SIZE > 1) it trains data-parallel, one process per GPU, like ``lcrec_b200.main``."""
import logging
import random

import numpy as np
import torch
from torch.utils.data import DataLoader

from ..datasets import EmbDataset
from ..main import build_parser, make_trainer
from .models.rqvae import RQVAE
from .trainer import DataParallelTrainer, Trainer


def parse_args(argv=None):
    p = build_parser("Index Training with Better Codebook Utilization")
    p.set_defaults(sk_epsilons=None)
    p.add_argument("--ema_decay", type=float, default=0.99)
    p.add_argument("--epsilon", type=float, default=1e-5)
    p.add_argument("--reset_threshold", type=float, default=1e-5)
    p.add_argument("--reset_interval", type=int, default=1000)
    return p.parse_args(argv)


def main(argv=None):
    seed = 2024
    random.seed(seed); np.random.seed(seed); torch.manual_seed(seed); torch.cuda.manual_seed_all(seed)
    args = parse_args(argv)
    print("=================================================")
    print("RQ-VAE Training with Better Codebook Utilization")
    print("=================================================")
    print(args)
    print("=================================================")
    print(f"EMA Decay: {args.ema_decay}")
    print(f"Reset Threshold: {args.reset_threshold}")
    print(f"Reset Interval: {args.reset_interval}")
    print("=================================================")
    logging.basicConfig(level=logging.DEBUG)
    data = EmbDataset(args.data_path)
    if args.sk_epsilons is None:
        args.sk_epsilons = [0.0] * len(args.num_emb_list)
    model = RQVAE(in_dim=data.dim, num_emb_list=args.num_emb_list, e_dim=args.e_dim, layers=args.layers,
                  dropout_prob=args.dropout_prob, bn=args.bn, loss_type=args.loss_type,
                  quant_loss_weight=args.quant_loss_weight, beta=args.beta, kmeans_init=args.kmeans_init,
                  kmeans_iters=args.kmeans_iters, sk_epsilons=args.sk_epsilons, sk_iters=args.sk_iters,
                  ema_decay=args.ema_decay, epsilon=args.epsilon, reset_threshold=args.reset_threshold,
                  reset_interval=args.reset_interval)
    print(model)
    loader = DataLoader(data, num_workers=args.num_workers, batch_size=args.batch_size, shuffle=True, pin_memory=True)
    best_loss, best_collision_rate = make_trainer(args, model, len(loader), Trainer, DataParallelTrainer).fit(loader)
    print("=================================================")
    print("Training Completed!")
    print(f"Best Loss: {best_loss}")
    print(f"Best Collision Rate: {best_collision_rate}")
    print("=================================================")


if __name__ == "__main__":
    main()
