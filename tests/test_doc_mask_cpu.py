"""Document masking without a GPU: native segment fill of the token loader, the masked reference attention math, document
independence, the GPT-2 graph with doc_mask, planner placement of the ids and distributed parity (gloo)."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from tepdist_b200.data import TokenLoader, segments_from_tokens, write_token_file  # noqa: E402
from tepdist_b200.ops.attention import attention_bwd, attention_fwd  # noqa: E402


# ------------------------------------------------------------------------------------------------ loader
def _packed(n, eot, seed, vocab=500):
    rng = np.random.default_rng(seed)
    a = rng.integers(0, vocab, n)
    a[rng.random(n) < 0.08] = eot
    return a


def test_segments_from_tokens_convention():
    tok = torch.tensor([[5, 9, 7, 9, 9, 1], [9, 9, 9, 9, 9, 9]])
    assert segments_from_tokens(tok, 9).tolist() == [[0, 0, 1, 1, 2, 3], [0, 1, 2, 3, 4, 5]]
    assert segments_from_tokens(tok, 9).dtype == torch.int32


@pytest.mark.parametrize("dtype", ["uint16", "int32"])
def test_native_segments_equal_segments_from_tokens(tmp_path, dtype):
    eot = 50256 if dtype == "uint16" else 70000
    path, bpt = write_token_file(str(tmp_path / "t.bin"), _packed(5000, eot, 0, vocab=eot), dtype)
    ld = TokenLoader(path, batch=3, n_ctx=64, seed=7, bytes_per_token=bpt, eot=eot, steps=5, pin=False, threads=3)
    n = 0
    for feeds in ld:
        assert set(feeds) == {"tokens", "labels", "segments"}
        assert torch.equal(feeds["segments"], segments_from_tokens(feeds["tokens"], eot))
        n += int(feeds["segments"].max())
    assert n > 0      # the windows really span several documents


def test_native_segments_with_a_mixture_and_resume(tmp_path):
    eot = 3
    a, bpa = write_token_file(str(tmp_path / "a.bin"), _packed(3000, eot, 1, vocab=50), "uint16")
    b, bpb = write_token_file(str(tmp_path / "b.bin"), _packed(3000, eot, 2, vocab=50), "uint16")
    kw = dict(batch=2, n_ctx=32, seed=1, mix=[(a, 1.0), (b, 3.0)], eot=eot, pin=False)
    full = [{k: v.clone() for k, v in f.items()} for f in TokenLoader(steps=6, **kw)]
    resumed = [{k: v.clone() for k, v in f.items()} for f in TokenLoader(steps=3, start_step=3, **kw)]
    for f in full:
        assert torch.equal(f["segments"], segments_from_tokens(f["tokens"], eot))
    for f, r in zip(full[3:], resumed):
        assert all(torch.equal(f[k], r[k]) for k in f)


def test_loader_without_eot_is_unchanged(tmp_path):
    path, bpt = write_token_file(str(tmp_path / "t.bin"), _packed(2000, 7, 3), "uint16")
    plain = [{k: v.clone() for k, v in f.items()} for f in TokenLoader(path, batch=2, n_ctx=16, steps=3, pin=False)]
    masked = [{k: v.clone() for k, v in f.items()} for f in TokenLoader(path, batch=2, n_ctx=16, steps=3, pin=False, eot=7)]
    for p, m in zip(plain, masked):
        assert set(p) == {"tokens", "labels"}
        assert torch.equal(p["tokens"], m["tokens"]) and torch.equal(p["labels"], m["labels"])


# ------------------------------------------------------------------------------------------------ reference math
def _dense(q, k, v, do, scale, mask):
    """Autograd attention with an explicit boolean mask [B, S, S] (rows without a visible key: o = 0)."""
    q, k, v = (t.detach().double().requires_grad_(True) for t in (q, k, v))
    s = torch.einsum("bqhd,bkhd->bhqk", q, k) * scale
    m = mask.unsqueeze(1)
    s = s.masked_fill(~m, float("-inf"))
    lse = torch.logsumexp(s, -1)
    p = torch.exp(s - lse.unsqueeze(-1)).masked_fill(~m, 0.0)
    o = torch.einsum("bhqk,bkhd->bqhd", p, v)
    o.backward(do.double())
    return o.detach(), lse.detach(), q.grad, k.grad, v.grad


def _layouts(B, S, g):
    one = torch.zeros(B, S, dtype=torch.int32)
    rnd = torch.stack([torch.cumsum((torch.rand(S, generator=g) < 0.05).int(), 0) for _ in range(B)]).int()
    single = torch.arange(S, dtype=torch.int32).repeat(B, 1) // 1          # every token its own document
    nonmono = torch.randint(0, 3, (B, S), generator=g, dtype=torch.int32) * 1000 - 1500
    ragged = (torch.arange(S) // 37).int().repeat(B, 1)                  # boundaries off the 128 grid
    return {"one": one, "random": rnd, "single_tokens": single, "non_monotone": nonmono, "off_grid": ragged}


@pytest.mark.parametrize("causal", [True, False])
@pytest.mark.parametrize("S", [64, 200])
def test_masked_reference_equals_dense_attention_with_an_explicit_mask(causal, S):
    g = torch.Generator().manual_seed(S + causal)
    B, H, D = 2, 2, 16
    q, k, v, do = (torch.randn(B, S, H, D, generator=g) for _ in range(4))
    scale = D ** -0.5
    for name, seg in _layouts(B, S, g).items():
        mask = seg[:, :, None] == seg[:, None, :]
        if causal:
            mask = mask & torch.ones(S, S, dtype=torch.bool).tril()
        o_r, lse_r, dq_r, dk_r, dv_r = _dense(q, k, v, do, scale, mask)
        o, lse = attention_fwd(q, k, v, scale, causal, seg_q=seg, seg_k=seg)
        assert torch.allclose(o.double(), o_r, atol=1e-5), name
        assert torch.allclose(lse.double(), lse_r, atol=1e-5), name
        dq, dk, dv = attention_bwd(do, q, k, v, o, lse, scale, causal, seg_q=seg, seg_k=seg)
        for a, b in ((dq, dq_r), (dk, dk_r), (dv, dv_r)):
            assert torch.allclose(a.double(), b, atol=1e-4), name


def test_rows_without_a_visible_key_give_zero_output_and_minus_inf_lse():
    B, S, H, D = 1, 32, 1, 8
    q, k, v = (torch.randn(B, S, H, D) for _ in range(3))
    sq, sk = torch.zeros(B, S, dtype=torch.int32), torch.ones(B, S, dtype=torch.int32)
    o, lse = attention_fwd(q, k, v, None, False, seg_q=sq, seg_k=sk)
    assert torch.all(o == 0) and torch.all(torch.isneginf(lse))
    dq, dk, dv = attention_bwd(torch.randn_like(q), q, k, v, o, lse, None, False, seg_q=sq, seg_k=sk)
    assert all(torch.all(t == 0) for t in (dq, dk, dv))


def test_document_independence_is_bit_exact():
    """Changing q / k / v / dO of document A leaves document B's o, lse and dq / dk / dv bit-identical: masked entries are exact
    zeros and never enter the row maximum."""
    g = torch.Generator().manual_seed(0)
    B, S, H, D = 1, 96, 2, 16
    seg = torch.tensor([[0] * 40 + [1] * 30 + [2] * 26], dtype=torch.int32)
    q, k, v, do = (torch.randn(B, S, H, D, generator=g) for _ in range(4))
    a = (seg == 1)[0]
    q2, k2, v2, do2 = (t.clone() for t in (q, k, v, do))
    for t in (q2, k2, v2, do2):
        t[:, a] = torch.randn(int(a.sum()), H, D, generator=g) * 30     # document A: large values change any shared maximum
    for causal in (True, False):
        o, lse = attention_fwd(q, k, v, None, causal, seg_q=seg)
        o2, lse2 = attention_fwd(q2, k2, v2, None, causal, seg_q=seg)
        gr = attention_bwd(do, q, k, v, o, lse, None, causal, seg_q=seg)
        gr2 = attention_bwd(do2, q2, k2, v2, o2, lse2, None, causal, seg_q=seg)
        keep = ~a
        assert torch.equal(o[:, keep], o2[:, keep]) and torch.equal(lse[:, :, keep], lse2[:, :, keep])
        for x, y in zip(gr, gr2):
            assert torch.equal(x[:, keep], y[:, keep])


# ------------------------------------------------------------------------------------------------ model and planner
def test_gpt2_doc_mask_with_one_document_equals_the_unmasked_model():
    from tepdist_b200.api import Trainer
    from tepdist_b200.models.gpt2 import CONFIGS, build_gpt2_graph
    cfg = CONFIGS["tiny"]
    torch.manual_seed(0)
    tok = torch.randint(0, cfg.n_vocab, (2, cfg.n_ctx), dtype=torch.int32)
    feeds = {"tokens": tok, "labels": torch.roll(tok, -1, 1)}
    losses = []
    for dm in (False, True):
        tr = Trainer(build_gpt2_graph(cfg, batch=2, doc_mask=dm), strategy="auto", device=torch.device("cpu"), use_cuda_graph=False)
        f = dict(feeds, segments=torch.zeros_like(tok)) if dm else feeds
        losses.append([tr.step(f) for _ in range(3)])
    assert losses[0] == losses[1], losses


def test_gpt2_doc_mask_graph_feeds_segments_to_every_attention_and_no_gradient():
    from tepdist_b200.models.gpt2 import CONFIGS, build_gpt2_graph
    g = build_gpt2_graph(CONFIGS["tiny"], batch=2, doc_mask=True)
    seg = next(n for n in g.nodes if n.op == "input" and n.name == "segments")
    att = [n for n in g.nodes if n.op in ("attention", "attention_bwd")]
    assert len(att) == 2 * CONFIGS["tiny"].n_layer
    assert all(n.inputs[-1].node == seg.id for n in att)
    users = {n.op for n in g.nodes if any(i.node == seg.id for i in n.inputs)}
    assert users == {"attention", "attention_bwd"}


# ------------------------------------------------------------------------------------------------ distributed (gloo)
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _run(cases, world, tmp_path, extra_env=None):
    out = str(tmp_path / f"doc_{world}_{len(cases)}.json")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", OMP_NUM_THREADS="2", **(extra_env or {}))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(HERE, "doc_mask_worker.py"), "+".join(cases), out]
    pr = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    assert pr.returncode == 0, pr.stderr[-3000:]
    return json.load(open(out))


_REF = {}


def _single():
    if "ref" not in _REF:
        import doc_mask_worker
        os.environ.pop("WORLD_SIZE", None)
        _REF["ref"] = doc_mask_worker.run("auto")
    return _REF["ref"]


def _check(got, ref, B=4, S=128):
    assert len(got["losses"]) == len(ref["losses"]) == 4        # (a fresh batch every step: the loss need not fall)
    for a, b in zip(got["losses"], ref["losses"]):
        assert abs(a - b) <= 2e-4 * max(1.0, abs(b)), (got, ref)
    shape = got["segments_shape"]
    assert shape[1] == S, got            # never split along the sequence
    assert shape[0] in (B, B // 2), got


_W2 = ["dp", "tp", "cp", "pp2m2"]


@pytest.fixture(scope="module")
def world2(tmp_path_factory):
    return _run(_W2, 2, tmp_path_factory.mktemp("w2"))


@pytest.mark.parametrize("strategy", _W2)
def test_doc_mask_world2_matches_single_process_and_keeps_segments_whole_along_the_sequence(world2, strategy):
    got, ref = world2[strategy], _single()
    _check(got, ref)
    par = got["parallelism"]
    if strategy == "dp":
        assert par.startswith("dp2") and got["segments_shape"] == [2, 128], got
    if strategy == "tp":
        assert par.startswith("tp") and got["segments_shape"] == [4, 128], got
    if strategy == "cp":
        assert par == "cp2" and got["segments_shape"] == [4, 128], got
    if strategy == "pp2m2":
        assert par.startswith("pp2"), got


def test_doc_mask_context_parallel_zigzag_matches_single_process(tmp_path):
    got = _run(["cp"], 2, tmp_path, {"TEPDIST_CP_ZIGZAG": "1"})["cp"]
    assert got["parallelism"] == "cp2"
    _check(got, _single())
    assert got["segments_shape"] == [4, 128], got


def test_doc_mask_dp2cp2_matches_single_process(tmp_path):
    got = _run(["dp2cp2"], 4, tmp_path)["dp2cp2"]
    _check(got, _single())      # (the data-parallel level may feed the ids whole and slice the batch locally)


def test_ring_block_interval_test_and_id_slices():
    """The interval test that decides which ring block products run (the products themselves run in the gloo cases)."""
    from tepdist_b200.parallel.ring_attention import RingAttention
    seg = torch.tensor([[0] * 16 + [1] * 16 + [1] * 16 + [2] * 16], dtype=torch.int32)
    s = RingAttention._Seg(seg, 4)
    assert s.meets(1, 2) and not s.meets(0, 1) and not s.meets(3, 0) and s.meets(0, 0)
    assert torch.equal(s.ids(3, 0), torch.cat((seg[:, 48:], seg[:, :16]), 1))
