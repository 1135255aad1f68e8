"""GPT-2 (the reference's headline example, examples/GPT2/models/gpt2/gpt2.py + *.json) expressed in
planner IR.  Structure follows SURVEY Appendix C: pre-LN blocks, tanh-GELU MLP (4x), separate untied LM
head, learned positions, no dropout (the reference's dropout is a no-op), AdamW; Q/K/V projections are
fused into one [3C, C] matmul (same math as the reference's three conv1d's).  The vocabulary is padded to
a multiple of 128 for the tensor-core tile; padded logits are masked inside the fused loss kernel.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

from ..frontend.builder import GraphBuilder, build_training_step
from ..ir import Graph


@dataclass
class GPT2Config:
    n_layer: int = 24
    n_embd: int = 1024
    n_head: int = 16
    n_ctx: int = 1024
    n_vocab: int = 50257
    batch: int = 4
    lr: float = 1e-4
    weight_decay: float = 0.01
    name: str = "gpt2-345M"

    @property
    def padded_vocab(self) -> int:
        return (self.n_vocab + 127) // 128 * 128

    def num_params(self) -> int:
        C, L, V = self.n_embd, self.n_layer, self.padded_vocab
        return 2 * V * C + self.n_ctx * C + L * (12 * C * C + 13 * C) + 2 * C

    def flops_per_token(self) -> float:
        C, L, V, S = self.n_embd, self.n_layer, self.padded_vocab, self.n_ctx
        dense = 6.0 * (L * 12 * C * C + V * C)
        attn = 6.0 * L * 2 * S * C / 2  # causal
        return dense + attn


CONFIGS = {
    "117M": GPT2Config(12, 768, 12, 1024, 50257, 4, name="gpt2-117M"),
    "345M": GPT2Config(24, 1024, 16, 1024, 50257, 4, name="gpt2-345M"),
    "1.5B": GPT2Config(48, 1600, 25, 1024, 50257, 4, name="gpt2-1.5B"),
    # examples/GPT2/PrettyBig.json, 175B.json (structural fields as given there, including the 175B file's n_ctx = 12288)
    "PrettyBig": GPT2Config(25, 1024, 16, 1024, 50257, 4, lr=2.5e-4, name="gpt2-PrettyBig"),
    "175B": GPT2Config(96, 12288, 96, 12288, 50257, 4, lr=2.5e-4, name="gpt2-175B"),
    "tiny": GPT2Config(2, 128, 2, 128, 1000, 2, name="gpt2-tiny"),
}


def build_gpt2_graph(cfg: GPT2Config, batch: int | None = None, optimizer: str = "adamw", doc_mask: bool = False,
                     **opt_hp) -> Graph:
    """`doc_mask=True`: a third input "segments" (int32 [B, n_ctx] document ids, e.g. `TokenLoader(..., eot=50256)` or
    `data.segments_from_tokens`) keeps every layer's attention inside each packed document."""
    B = batch or cfg.batch
    S, C, H, V, Vp = cfg.n_ctx, cfg.n_embd, cfg.n_head, cfg.n_vocab, cfg.padded_vocab
    b = GraphBuilder(cfg.name)
    tokens = b.input("tokens", (B, S), "i32")
    labels = b.input("labels", (B, S), "i32")
    segments = b.input("segments", (B, S), "i32") if doc_mask else None
    nrm = lambda std: {"kind": "normal", "mean": 0.0, "std": std}
    const = lambda v: {"kind": "constant", "value": v}
    with b.scope("model"):
        wte = b.parameter("wte", (Vp, C), nrm(0.02))
        wpe = b.parameter("wpe", (S, C), nrm(0.01))
        x = b.embedding(tokens, wte, wpe)
        for l in range(cfg.n_layer):
            with b.scope(f"h{l}"):
                g1 = b.parameter("ln_1/g", (C,), const(1.0)); b1 = b.parameter("ln_1/b", (C,), const(0.0))
                h = b.layernorm(x, g1, b1, name="ln_1")
                w_qkv = b.parameter("attn/c_attn/w", (3 * C, C), nrm(0.02)); b_qkv = b.parameter("attn/c_attn/b", (3 * C,), const(0.0))
                qkv = b.linear(h, w_qkv, b_qkv, name="attn/c_attn")
                a = b.attention(qkv, heads=H, causal=True, segments=segments, name="attn/core")
                w_o = b.parameter("attn/c_proj/w", (C, C), nrm(0.02 / math.sqrt(2 * cfg.n_layer))); b_o = b.parameter("attn/c_proj/b", (C,), const(0.0))
                x = b.linear(a, w_o, b_o, residual=x, name="attn/c_proj")
                g2 = b.parameter("ln_2/g", (C,), const(1.0)); b2 = b.parameter("ln_2/b", (C,), const(0.0))
                h = b.layernorm(x, g2, b2, name="ln_2")
                w_fc = b.parameter("mlp/c_fc/w", (4 * C, C), nrm(0.02)); b_fc = b.parameter("mlp/c_fc/b", (4 * C,), const(0.0))
                f = b.linear(h, w_fc, b_fc, name="mlp/c_fc")
                f = b.gelu(f, name="mlp/gelu")
                w_p = b.parameter("mlp/c_proj/w", (C, 4 * C), nrm(0.02 / math.sqrt(2 * cfg.n_layer))); b_p = b.parameter("mlp/c_proj/b", (C,), const(0.0))
                x = b.linear(f, w_p, b_p, residual=x, name="mlp/c_proj")
        gf = b.parameter("ln_f/g", (C,), const(1.0)); bf = b.parameter("ln_f/b", (C,), const(0.0))
        h = b.layernorm(x, gf, bf, name="ln_f")
        w_out = b.parameter("output", (Vp, C), nrm(0.02))
        logits = b.linear(h, w_out, name="lm_head")
        loss = b.softmax_xent(logits, labels, vocab=V, name="loss")
    g = build_training_step(b, loss, optimizer, **{**dict(lr=cfg.lr, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=cfg.weight_decay),
                                                     **opt_hp})      # (opt_hp: clip_norm / clip_norm_value / schedule / ...)
    g.meta["model"] = {"family": "gpt2", "name": cfg.name, "n_layer": cfg.n_layer, "n_embd": C, "n_head": H,
                       "n_ctx": S, "n_vocab": V, "batch": B, "doc_mask": bool(doc_mask)}
    return g
