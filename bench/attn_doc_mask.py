#!/usr/bin/env python
"""Document-masked attention on one GPU: masked forward + backward against the unmasked causal kernel, and a GPT-2 training step
with and without document masking.

    python bench/attn_doc_mask.py [--out results.json] [--skip-step]

Kernel part: B = 4, H = 16, D = 64, S in {1024, 8192} (qkv is 805 MB at S = 8192, well above the 126 MB L2; at S = 1024 it is
100 MB and stays L2-resident between passes).  Layouts: one document, 8 documents of S / 8 tokens, random lengths (mean S / 8).
The unmasked causal call and the masked call alternate inside one process (CUDA events around `--iters` fwd + bwd pairs,
median of `--reps` alternations, after warm-up).  Next to the times: the (query block, key block) pairs the masked kernels visit
against the causal count, computed from the ids exactly as the kernels decide.

Step part: GPT-2 345M, batch 4, n_ctx 1024, one GPU, packed synthetic tokens whose documents have a mean length of n_ctx / 4;
median step time over `--steps` steps with doc_mask False / True.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

EOT = 50256


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e!r})"


def layouts(B, S, g):
    docs = S // 8
    rnd = []
    for _ in range(B):
        ends = torch.rand(S, generator=g) < 1.0 / docs
        rnd.append(torch.cumsum(ends.int(), 0) - ends.int())
    return {"one_doc": torch.zeros(B, S, dtype=torch.int32),
            "8_docs": (torch.arange(S) // docs).int().repeat(B, 1),
            "random": torch.stack(rnd).int()}


def visited_pairs(seg, causal=True):
    """(query block, key block) pairs with overlapping id intervals, summed over the batch (per head)."""
    B, S = seg.shape
    v = seg.view(B, S // 128, 128)
    mn, mx = v.amin(2), v.amax(2)
    meet = (mn[:, :, None] <= mx[:, None, :]) & (mn[:, None, :] <= mx[:, :, None])
    if causal:
        meet &= torch.ones(S // 128, S // 128, dtype=torch.bool).tril()
    return int(meet.sum())


def time_pairs(fns, iters, reps):
    """Alternates the callables; returns the median ms per call of each."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in fns]
    ts = [[] for _ in fns]
    for _ in range(reps):
        for i, f in enumerate(fns):
            ev[i][0].record()
            for _ in range(iters):
                f()
            ev[i][1].record()
        torch.cuda.synchronize()
        for i in range(len(fns)):
            ts[i].append(ev[i][0].elapsed_time(ev[i][1]) / iters)
    return [statistics.median(t) for t in ts]


def kernels(iters, reps):
    from tepdist_b200 import ops
    B, H, D = 4, 16, 64
    res = []
    g = torch.Generator().manual_seed(0)
    for S in (1024, 8192):
        qkv = torch.randn(B, S, H, 3, D, device="cuda").to(torch.bfloat16)
        q, k, v = qkv[:, :, :, 0], qkv[:, :, :, 1], qkv[:, :, :, 2]
        do = torch.randn(B, S, H, D, device="cuda").to(torch.bfloat16)
        causal_pairs = B * (S // 128) * (S // 128 + 1) // 2

        def plain():
            o, lse = ops.attention_fwd(q, k, v, causal=True)
            ops.attention_bwd(do, q, k, v, o, lse, causal=True)

        for name, seg in layouts(B, S, g).items():
            sd = seg.cuda()

            def masked():
                o, lse = ops.attention_fwd(q, k, v, causal=True, seg_q=sd, seg_k=sd)
                ops.attention_bwd(do, q, k, v, o, lse, causal=True, seg_q=sd, seg_k=sd)

            def masked_fwd():
                ops.attention_fwd(q, k, v, causal=True, seg_q=sd, seg_k=sd)

            def plain_fwd():
                ops.attention_fwd(q, k, v, causal=True)

            for f in (plain, masked, plain_fwd, masked_fwd):
                for _ in range(3):
                    f()
            torch.cuda.synchronize()
            t_plain, t_masked = time_pairs([plain, masked], iters, reps)
            t_pf, t_mf = time_pairs([plain_fwd, masked_fwd], iters, reps)
            vp = visited_pairs(seg)
            r = {"S": S, "layout": name, "docs_mean_len": float(S * B / (int(seg.max(1).values.sum()) + B)),
                 "causal_ms": round(t_plain, 4), "masked_ms": round(t_masked, 4), "time_ratio": round(t_masked / t_plain, 4),
                 "causal_fwd_ms": round(t_pf, 4), "masked_fwd_ms": round(t_mf, 4), "fwd_time_ratio": round(t_mf / t_pf, 4),
                 "visited_pairs": vp, "causal_pairs": causal_pairs, "pair_ratio": round(vp / causal_pairs, 4)}
            print(json.dumps(r), flush=True)
            res.append(r)
        del qkv, q, k, v, do
        torch.cuda.empty_cache()
    return res


def packed_tokens(B, S, mean_doc, vocab, g):
    tok = torch.randint(0, vocab - 1, (B, S), generator=g, dtype=torch.int32)
    tok[torch.rand(B, S, generator=g) < 1.0 / mean_doc] = EOT
    return tok


def step_times(steps):
    from tepdist_b200.api import Trainer
    from tepdist_b200.data import segments_from_tokens
    from tepdist_b200.models.gpt2 import CONFIGS, build_gpt2_graph
    import time
    cfg = CONFIGS["345M"]
    g = torch.Generator().manual_seed(0)
    tok = packed_tokens(cfg.batch, cfg.n_ctx, cfg.n_ctx // 4, cfg.n_vocab, g)
    feeds = {"tokens": tok, "labels": torch.roll(tok, -1, 1)}
    out = {}
    for dm in (False, True):
        tr = Trainer(build_gpt2_graph(cfg, doc_mask=dm), strategy="auto")
        f = dict(feeds, segments=segments_from_tokens(tok, EOT)) if dm else feeds
        for _ in range(3):
            tr.step(f)
        ts = []
        for _ in range(steps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            loss = tr.step(f)
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
        out["doc_mask" if dm else "causal"] = {"median_ms": round(statistics.median(ts), 3), "min_ms": round(min(ts), 3),
                                               "loss": float(loss)}
        print(json.dumps({"step": "doc_mask" if dm else "causal", **out["doc_mask" if dm else "causal"]}), flush=True)
        del tr
        torch.cuda.empty_cache()
    segs = segments_from_tokens(tok, EOT)
    out["mean_doc_len"] = float(tok.numel() / (int(segs.max(1).values.sum()) + tok.shape[0]))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--steps", type=int, default=15)
    ap.add_argument("--skip-step", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a GPU")
    res = {"card": card(), "kernels": kernels(a.iters, a.reps)}
    if not a.skip_step:
        res["gpt2_345M_step"] = step_times(a.steps)
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
