"""Worker for the document-masking parity tests: python tests/doc_mask_worker.py <strategy[+strategy...]> <out.json> under torchrun
(gloo on CPU; TEPDIST_TEST_DEVICE=cuda runs over NCCL on GPUs).  GPT-2 with doc_mask=True trained for a few steps on a packed
token file whose documents are shorter than n_ctx; reports the losses and the local shape of the "segments" input."""
import dataclasses
import json
import os
import sys
import tempfile

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

EOT = 999      # inside the tiny config's vocabulary of 1000


def packed_token_file(path, n_tokens=20000, mean_doc=40, seed=1):
    """Documents of random length (mean `mean_doc`), each closed by EOT."""
    from tepdist_b200.data import write_token_file
    rng = np.random.default_rng(seed)
    out = []
    while len(out) < n_tokens:
        n = int(rng.integers(1, 2 * mean_doc))
        out.extend(rng.integers(0, EOT, n).tolist())
        out.append(EOT)
    return write_token_file(path, out[:n_tokens])


def _dev():
    if os.environ.get("TEPDIST_TEST_DEVICE") == "cuda":
        return torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    return torch.device("cpu")


def _segments_shape(tr):
    graphs = [getattr(tr.exec, "g", None)]
    worker = getattr(tr.exec, "worker", None)
    if worker is not None:
        graphs.append(worker.sub)
    for g in graphs:
        for n in getattr(g, "nodes", []):
            if n.op == "input" and n.name == "segments":
                return list(n.outputs[0].shape)
    return None


def run(strategy, n_ctx=None, steps=4):
    from tepdist_b200.api import Trainer
    from tepdist_b200.data import TokenLoader
    from tepdist_b200.models.gpt2 import CONFIGS, build_gpt2_graph
    cfg = CONFIGS["tiny"]
    if n_ctx or os.environ.get("TEPDIST_TEST_NCTX"):
        cfg = dataclasses.replace(cfg, n_ctx=int(n_ctx or os.environ["TEPDIST_TEST_NCTX"]))
    if int(os.environ.get("WORLD_SIZE", "1")) == 1:
        strategy = "auto"            # single-process oracle
    g = build_gpt2_graph(cfg, batch=4, doc_mask=True)
    tr = Trainer(g, strategy=strategy, device=_dev(), use_cuda_graph=False)
    with tempfile.TemporaryDirectory() as d:
        path, bpt = packed_token_file(os.path.join(d, "docs.bin"))
        loader = TokenLoader(path, batch=4, n_ctx=cfg.n_ctx, seed=3, bytes_per_token=bpt, eot=EOT, steps=steps, pin=False)
        losses = []
        for feeds in loader:
            losses.append(tr.step({k: v.clone() for k, v in feeds.items()}))
    return {"losses": losses, "parallelism": tr.plan_info.get("parallelism"), "segments_shape": _segments_shape(tr),
            "n_ctx": cfg.n_ctx}


if __name__ == "__main__":
    cases, out = sys.argv[1], sys.argv[2]
    res = {c: run(c) for c in cases.split("+")}
    if int(os.environ.get("RANK", "0")) == 0:
        json.dump(res, open(out, "w"))
    if dist.is_initialized():
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
