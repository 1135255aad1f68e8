"""Input pipeline: token files -> {"tokens", "labels"} batches in pinned host memory, prefetched by native threads.

The reference's client feeds its examples through tf.data (examples/GPT2/inputs.py: BPE token records, windows of n_ctx + 1
tokens split into input / next-token label, datasets mixed by weight, prefetch, and a random-token `fake_input` mode).  This
module offers the same through `_C.TokenSource` / `_C.BatchLoader` (csrc/runtime/data_loader.cc):

    loader = TokenLoader(["shard0.bin", "shard1.bin"], batch=4, n_ctx=1024, rank=tr.rank, world=tr.world, seed=0)
    for feeds in loader:                 # {"tokens": int32 [batch, n_ctx], "labels": int32 [batch, n_ctx]} -- THIS rank's rows
        loss = tr.step(feeds)

* Files are flat little-endian uint16 (vocab < 65536) or int32 token streams (`write_token_file`), memory-mapped.
* Sampling is stateless: sample k of the run is a pure function of (seed, k); rank r of `world` takes rows
  [r * batch, (r + 1) * batch) of global batch t.  No coordination between ranks, and `start_step=k` resumes a stream exactly.
* `prefetch` slots of page-locked memory are filled ahead by `threads` native threads; a yielded batch stays valid until the next
  one is requested (the training step's host->device copy reads straight from it).
* `mix=[(files, weight), ...]`: several datasets sampled by weight; `synthetic_vocab=V`: random tokens (the reference's fake_input).
* `eot=50256`: batches also carry "segments", int32 [batch, n_ctx] document ids for document-masked attention
  (`build_gpt2_graph(..., doc_mask=True)`), filled by the same native threads: `segments_from_tokens(tokens, eot)`.
"""
from __future__ import annotations

from typing import Dict, Iterator, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

Files = Union[str, Sequence[str]]


def write_token_file(path: str, tokens, dtype: str = "auto") -> Tuple[str, int]:
    """Write a flat token stream.  dtype 'uint16' | 'int32' | 'auto' (uint16 when every id fits).  Returns (path, bytes per token)."""
    a = np.asarray(tokens).reshape(-1)
    if dtype == "auto":
        dtype = "uint16" if a.size == 0 or (int(a.min()) >= 0 and int(a.max()) < 65536) else "int32"
    if dtype not in ("uint16", "int32"):
        raise ValueError("dtype must be 'uint16', 'int32' or 'auto'")
    a.astype("<u2" if dtype == "uint16" else "<i4").tofile(path)
    return path, 2 if dtype == "uint16" else 4


def segments_from_tokens(tokens: torch.Tensor, eot: int) -> torch.Tensor:
    """Document ids of packed windows [..., n]: seg[i] = number of `eot` tokens at positions < i along the last dim, so the
    end-of-text token belongs to the document it ends.  int32, on the device of `tokens` (CPU or CUDA)."""
    ends = (tokens == eot).to(torch.int32)
    seg = torch.cumsum(ends, -1, dtype=torch.int32) - ends
    return seg


class TokenLoader:
    """Iterator over this rank's batches; see the module docstring."""

    def __init__(self, files: Optional[Files] = None, *, batch: int, n_ctx: int, rank: int = 0, world: int = 1, seed: int = 0,
                 mix: Optional[Sequence[Tuple[Files, float]]] = None, synthetic_vocab: int = 0, bytes_per_token: int = 2,
                 prefetch: int = 4, threads: int = 2, start_step: int = 0, steps: Optional[int] = None, pin: Optional[bool] = None,
                 eot: Optional[int] = None):
        from .. import _C
        if sum(x is not None and x != 0 for x in (files, mix, synthetic_vocab)) != 1:
            raise ValueError("give exactly one of files=, mix= or synthetic_vocab=")
        self.source = _C.TokenSource()
        if synthetic_vocab:
            self.source.set_synthetic(int(synthetic_vocab))
        else:
            for fs, w in (mix if mix is not None else [(files, 1.0)]):
                self.source.add_dataset([fs] if isinstance(fs, str) else list(fs), float(w), int(bytes_per_token))
        self.batch, self.n_ctx, self.rank, self.world, self.seed = int(batch), int(n_ctx), int(rank), int(world), int(seed)
        self.steps = steps
        pin = torch.cuda.is_available() if pin is None else pin
        mk = lambda: torch.empty(self.batch, self.n_ctx, dtype=torch.int32, pin_memory=bool(pin))
        self._tok: List[torch.Tensor] = [mk() for _ in range(max(2, int(prefetch)))]
        self._lab: List[torch.Tensor] = [mk() for _ in range(len(self._tok))]
        self._loader = _C.BatchLoader(self.source, self.batch, self.n_ctx, self.rank, self.world, self.seed, int(threads))
        self.eot = None if eot is None else int(eot)
        self._seg: List[torch.Tensor] = [mk() for _ in range(len(self._tok))] if self.eot is not None else []
        self._loader.set_buffers([t.data_ptr() for t in self._tok], [t.data_ptr() for t in self._lab],
                                 [t.data_ptr() for t in self._seg], 0 if self.eot is None else self.eot)
        self._held: Optional[int] = None
        self.step = int(start_step)          # step of the NEXT batch
        self._first = int(start_step)
        self._loader.start(self.step)

    def __iter__(self) -> Iterator[Dict[str, torch.Tensor]]:
        return self

    def __next__(self) -> Dict[str, torch.Tensor]:
        if self.steps is not None and self.step - self._first >= self.steps:
            self.close()
            raise StopIteration
        if self._held is not None:
            self._loader.release(self._held)        # the previous batch's buffers go back to the workers
        slot, step = self._loader.acquire()
        assert step == self.step, (step, self.step)
        self._held = slot
        self.step += 1
        if self.eot is not None:
            return {"tokens": self._tok[slot], "labels": self._lab[slot], "segments": self._seg[slot]}
        return {"tokens": self._tok[slot], "labels": self._lab[slot]}

    def close(self) -> None:
        if self._loader is not None:
            self._loader.stop()
            self._loader = None
            self._held = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ introspection (tests, debugging)
    def sample(self, sample_id: int) -> torch.Tensor:
        """The n_ctx + 1 tokens of global sample `sample_id` (what row (sample_id % global_batch) of step sample_id // global_batch holds)."""
        return torch.tensor(self.source.sample(self.seed, int(sample_id), self.n_ctx + 1), dtype=torch.int32)
