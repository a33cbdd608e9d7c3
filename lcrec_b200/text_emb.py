"""Embedding producer hand-off (SURVEY 8(f) rank 4): ``generate_item_embedding`` with the signature and file contract of
reference ``data_process/amazon_text_emb.py:49-105``.

The tokenizer and the PLM are the caller's (Hugging Face objects; the PLM forward is outside this library's scope).  What
happens to ``outputs.last_hidden_state`` is ours: the masked mean pool (:91-92) and the mean over the item's text fields
(:96) run in ``lcrec_masked_mean_pool`` and write straight into the rows of ONE fp32 (N, hidden) device matrix - the matrix
``Indexer.run`` / ``lcrec_indexer_run_device`` reads - instead of a Python list of CPU tensors, a ``torch.cat`` and an
``.npy`` round trip.  The ``.npy`` file of the reference (``<root>/<dataset>.emb-<plm_name>-td.npy``, :104-105) is still
written unless ``save=False``; the device matrix is returned.

``dtype=torch.float16`` / ``torch.bfloat16`` keeps the matrix in half precision (half the memory, and the indexer reads it
without an fp32 copy): each batch is pooled into an fp32 scratch of ``batch_size`` rows as above and rounded once into its
rows, so the matrix equals the fp32 one ``.to(dtype)``.  An fp16 matrix is saved as an fp16 ``.npy``; numpy has no bf16.
"""
from __future__ import annotations

import os
import random

import numpy as np
import torch

from . import ops


@torch.no_grad()
def generate_item_embedding(args, item_text_list, tokenizer, model, word_drop_ratio=-1, batch_size=1, save=True,
                            dtype=torch.float32):
    """args: .root, .dataset, .plm_name, .max_sent_len, .device (a CUDA device).  Returns the (N, hidden) device matrix of
    ``dtype`` (fp32, fp16 or bf16).  ``batch_size`` 1 is the reference's hard-coded value (:61); larger batches pool several
    items per launch."""
    if dtype not in (torch.float32, torch.float16, torch.bfloat16):
        raise ValueError(f"generate_item_embedding: dtype must be float32, float16 or bfloat16, not {dtype}")
    if save and dtype == torch.bfloat16:
        raise ValueError("generate_item_embedding: numpy has no bfloat16, so a bf16 matrix cannot be saved as .npy "
                         "(use save=False, or dtype=torch.float16)")
    print("Generate Text Embedding: ")
    print(" Dataset: ", args.dataset)
    items, texts = zip(*item_text_list)
    order_texts = [[0]] * len(items)
    for item, text in zip(items, texts):
        order_texts[item] = text
    for text in order_texts:
        assert text != [0]

    embeddings = scratch = None
    start = 0
    while start < len(order_texts):
        if (start + 1) % 100 == 0:
            print("==>", start + 1)
        batch = order_texts[start: start + batch_size]
        fields = [list(sentences) for sentences in zip(*batch)]
        for f, sentences in enumerate(fields):
            if word_drop_ratio > 0:                       # :73-85, same draws from Python's RNG
                print(f"Word drop with p={word_drop_ratio}")
                kept = []
                for sent in sentences:
                    kept.append(" ".join(wd for wd in sent.split(" ") if random.random() > word_drop_ratio))
                sentences = kept
            enc = tokenizer(sentences, max_length=args.max_sent_len, truncation=True, return_tensors="pt",
                            padding="longest").to(args.device)
            outputs = model(input_ids=enc.input_ids, attention_mask=enc.attention_mask)
            h = outputs.last_hidden_state
            if embeddings is None:
                embeddings = torch.empty((len(order_texts), h.shape[-1]), dtype=dtype, device=h.device)
                if dtype != torch.float32:
                    scratch = torch.empty((batch_size, h.shape[-1]), dtype=torch.float32, device=h.device)
            rows = embeddings[start: start + len(batch)] if scratch is None else scratch[: len(batch)]
            ops.masked_mean_pool(h, enc["attention_mask"], out=rows, accumulate=f > 0,
                                 divide_by=float(len(fields)) if f == len(fields) - 1 else 0.0)
        if scratch is not None:
            embeddings[start: start + len(batch)].copy_(scratch[: len(batch)])      # one rounding to the half format
        start += batch_size
    print("Embeddings shape: ", tuple(embeddings.shape))
    if save:
        file = os.path.join(args.root, args.dataset + ".emb-" + args.plm_name + "-td" + ".npy")
        np.save(file, embeddings.cpu().numpy())
    return embeddings
