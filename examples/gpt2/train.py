#!/usr/bin/env python
"""GPT-2 training (reference examples/GPT2/main.py: "Train loop took X s").  Input: synthetic `fake_input` by default (one fixed
random batch, like the reference's FAKE_INPUT server flag), `--data a.bin,b.bin` for token files through the native prefetching
loader (tepdist_b200/data: memory-mapped uint16 / int32 token streams, windows of n_ctx + 1 tokens, stateless sampling), or
`--data synthetic` for a fresh random batch every step from the same loader."""
import argparse
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from tepdist_b200.api import Trainer  # noqa: E402
from tepdist_b200.models.gpt2 import CONFIGS, build_gpt2_graph  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", default="345M", choices=list(CONFIGS))
    ap.add_argument("--batch", type=int, default=4, help="sequences per GPU")
    ap.add_argument("--train-steps", type=int, default=10)
    ap.add_argument("--strategy", default="auto")
    ap.add_argument("--comm", default="fused", choices=["fused", "nccl"])
    ap.add_argument("--warmup-steps", type=int, default=0, help='linear warm-up then cosine decay over --train-steps (reference json: "warmup_steps")')
    ap.add_argument("--optimizer", default="adamw", choices=["adam", "adamw", "adafactor", "lamb", "sm3", "momentum", "sgd"],
                    help='reference: "opt_name" adam | adafactor in examples/GPT2/*.json')
    ap.add_argument("--clip-norm", default=None, choices=["global", "local"], help='gradient clipping (reference gpt_moe config: "clip_norm")')
    ap.add_argument("--clip-norm-value", type=float, default=1.0)
    ap.add_argument("--data", default=None, help="comma-separated token files (see tepdist_b200.data.write_token_file) or 'synthetic'")
    ap.add_argument("--data-int32", action="store_true", help="token files hold int32 ids (default uint16)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--doc-mask", action="store_true",
                    help="document masking: attention stays inside each document of a packed window (documents end at --eot)")
    ap.add_argument("--eot", type=int, default=50256, help="end-of-text token id that closes a document (GPT-2 BPE: 50256)")
    a = ap.parse_args()
    clip = {"clip_norm": a.clip_norm, "clip_norm_value": a.clip_norm_value} if a.clip_norm else {}
    cfg = CONFIGS[a.model]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    g = build_gpt2_graph(cfg, batch=a.batch * world, optimizer=a.optimizer, doc_mask=a.doc_mask, **clip)
    tr = Trainer(g, strategy=a.strategy, comm_mode=a.comm)
    if a.warmup_steps > 0:
        from tepdist_b200.utils.schedules import warmup_cosine
        tr.set_lr_schedule(warmup_cosine(cfg.lr, a.warmup_steps, a.train_steps))
    if a.data:
        # every rank draws the same GLOBAL batch (sampling is a pure function of seed and step) and the trainer takes the rows /
        # columns its plan assigns to this rank: works unchanged under data, tensor, context and pipeline parallel plans
        from tepdist_b200.data import TokenLoader
        src = {"synthetic_vocab": cfg.n_vocab} if a.data == "synthetic" else {"files": a.data.split(","), "bytes_per_token": 4 if a.data_int32 else 2}
        batches = iter(TokenLoader(batch=a.batch * world, n_ctx=cfg.n_ctx, seed=a.seed, eot=a.eot if a.doc_mask else None, **src))
    else:
        gen = torch.Generator().manual_seed(a.seed)
        tok = torch.randint(0, cfg.n_vocab, (a.batch * world, cfg.n_ctx), generator=gen, dtype=torch.int32)
        fixed = {"tokens": tok, "labels": torch.roll(tok, -1, 1)}
        if a.doc_mask:
            from tepdist_b200.data import segments_from_tokens
            fixed["segments"] = segments_from_tokens(tok, a.eot)
        batches = iter(lambda: fixed, None)
    t0 = time.time()
    for i in range(a.train_steps):
        loss = tr.step(next(batches))
        if tr.rank == 0:
            print(f"step {i} loss {loss:.4f}")
    if tr.rank == 0:
        dt = time.time() - t0
        print(f"Train loop took {dt:.2f} s  ({a.train_steps * a.batch * world * cfg.n_ctx / dt:.0f} tokens/s incl. planning + warm-up); "
              f"plan: {tr.plan_info.get('parallelism', 'single')}")
    os._exit(0)


if __name__ == "__main__":
    main()
