"""Document-masked attention on the B200: the SEG instantiations of the tcgen05 forward / backward kernels against the fp32
reference, bit-identity with the unmasked kernels for one document, document independence, empty ring blocks, CUDA-graph
replay, and GPT-2 training with doc_mask on one GPU (against the CPU) and under cp2 on two GPUs (against one GPU)."""
import json
import os
import socket
import subprocess
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

pytestmark = pytest.mark.gpu


def _qkv(B, S, H, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    qkv = torch.randn(B, S, H, 3, 64, device="cuda", generator=g).to(torch.bfloat16)
    return qkv, qkv[:, :, :, 0], qkv[:, :, :, 1], qkv[:, :, :, 2]


def _rel(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm().clamp_min(1e-12)).item()


def _layouts(B, S):
    g = torch.Generator().manual_seed(S)
    lens = lambda: torch.cumsum((torch.rand(S, generator=g) < 3.0 / 512).int(), 0)      # random lengths, mean ~170 tokens
    return {
        "one": torch.zeros(B, S, dtype=torch.int32),
        "random": torch.stack([lens() for _ in range(B)]).int(),
        "aligned128": (torch.arange(S) // 256).int().repeat(B, 1),
        "non_monotone": (torch.randint(0, 4, (B, S // 64), generator=g).repeat_interleave(64, 1) * 7 - 9).int(),
    }


def _reference(q, k, v, do, seg, causal):
    S = q.shape[1]
    qr, kr, vr = (t.float().detach().clone().requires_grad_(True) for t in (q, k, v))
    s = torch.einsum("bqhd,bkhd->bhqk", qr, kr) / 8.0
    m = (seg[:, :, None] == seg[:, None, :]).unsqueeze(1)
    if causal:
        m = m & torch.ones(S, S, dtype=torch.bool, device="cuda").tril()
    s = s.masked_fill(~m, float("-inf"))
    lse = torch.logsumexp(s, -1)
    o = torch.einsum("bhqk,bkhd->bqhd", torch.exp(s - lse.unsqueeze(-1)).masked_fill(~m, 0.0), vr)
    o.backward(do.float())
    return o.detach(), lse.detach(), qr.grad, kr.grad, vr.grad


@pytest.mark.parametrize("S", [1024, 4096])
def test_masked_kernels_match_the_fp32_reference(S):
    from tepdist_b200 import ops
    B, H = 4, 16
    qkv, q, k, v = _qkv(B, S, H)
    do = torch.randn(B, S, H, 64, device="cuda").to(torch.bfloat16)
    cases = [(name, seg, True) for name, seg in _layouts(B, S).items()] + [("random_noncausal", _layouts(B, S)["random"], False)]
    for name, seg, causal in cases:
        seg = seg.cuda()
        n0 = ops.launch_count()
        o, lse = ops.attention_fwd(q, k, v, causal=causal, seg_q=seg, seg_k=seg)
        dq, dk, dv = ops.attention_bwd(do, q, k, v, o, lse, causal=causal, seg_q=seg, seg_k=seg)
        torch.cuda.synchronize()
        assert ops.launch_count() - n0 == 6                      # pre-pass + forward, pre-pass + delta + backward + dq cast
        o_r, lse_r, dq_r, dk_r, dv_r = _reference(q, k, v, do, seg, causal)
        err = {"o": _rel(o, o_r), "lse": _rel(lse, lse_r), "dq": _rel(dq, dq_r), "dk": _rel(dk, dk_r), "dv": _rel(dv, dv_r)}
        assert err["o"] < 2e-2 and err["lse"] < 1e-3 and max(err["dq"], err["dk"], err["dv"]) < 3e-2, (name, err)
        assert not any(torch.isnan(t).any() for t in (o, lse, dq, dk, dv)), name
        del o_r, lse_r, dq_r, dk_r, dv_r


def test_one_document_is_bit_identical_to_the_unmasked_causal_kernel():
    from tepdist_b200 import ops
    B, H, S = 4, 16, 1024
    qkv, q, k, v = _qkv(B, S, H, seed=1)
    do = torch.randn(B, S, H, 64, device="cuda").to(torch.bfloat16)
    seg = torch.full((B, S), 5, dtype=torch.int32, device="cuda")
    o0, l0 = ops.attention_fwd(q, k, v, causal=True)
    o1, l1 = ops.attention_fwd(q, k, v, causal=True, seg_q=seg, seg_k=seg)
    g0 = ops.attention_bwd(do, q, k, v, o0, l0, causal=True)
    g0 = [t.clone() for t in g0]
    g1 = ops.attention_bwd(do, q, k, v, o1, l1, causal=True, seg_q=seg, seg_k=seg)
    torch.cuda.synchronize()
    assert torch.equal(o0, o1) and torch.equal(l0, l1)
    assert torch.equal(g0[1], g1[1]) and torch.equal(g0[2], g1[2])            # dk, dv: one CTA each, fixed order
    assert _rel(g1[0], g0[0]) < 1e-2            # dq: fp32 red.add over key-block CTAs, order differs from run to run


def test_document_independence_on_the_device():
    from tepdist_b200 import ops
    B, H, S = 2, 4, 1024
    seg = torch.tensor([0] * 300 + [1] * 200 + [2] * 524, dtype=torch.int32, device="cuda").repeat(B, 1)
    qkv, q, k, v = _qkv(B, S, H, seed=2)
    do = torch.randn(B, S, H, 64, device="cuda").to(torch.bfloat16)
    a = seg[0] == 1
    qkv2, do2 = qkv.clone(), do.clone()
    qkv2[:, a] = (torch.randn_like(qkv2[:, a].float()) * 20).to(torch.bfloat16)
    do2[:, a] = torch.randn_like(do2[:, a])
    q2, k2, v2 = qkv2[:, :, :, 0], qkv2[:, :, :, 1], qkv2[:, :, :, 2]
    for causal in (True, False):
        o, l = ops.attention_fwd(q, k, v, causal=causal, seg_q=seg, seg_k=seg)
        o2, l2 = ops.attention_fwd(q2, k2, v2, causal=causal, seg_q=seg, seg_k=seg)
        g = [t.clone() for t in ops.attention_bwd(do, q, k, v, o, l, causal=causal, seg_q=seg, seg_k=seg)]
        g2 = ops.attention_bwd(do2, q2, k2, v2, o2, l2, causal=causal, seg_q=seg, seg_k=seg)
        torch.cuda.synchronize()
        keep = ~a
        assert torch.equal(o[:, keep], o2[:, keep]) and torch.equal(l[:, :, keep], l2[:, :, keep]), causal
        assert torch.equal(g[1][:, keep], g2[1][:, keep]) and torch.equal(g[2][:, keep], g2[2][:, keep]), causal
        assert _rel(g2[0][:, keep], g[0][:, keep]) < 1e-2, causal     # dq: atomic summation order only


def test_ring_block_with_disjoint_ids_is_empty():
    from tepdist_b200 import ops
    B, H, S = 2, 4, 256
    qkv, q, k, v = _qkv(B, S, H, seed=3)
    sq = torch.zeros(B, S, dtype=torch.int32, device="cuda")
    sk = torch.ones(B, S, dtype=torch.int32, device="cuda")
    o, lse = ops.attention_fwd(q, k, v, causal=False, seg_q=sq, seg_k=sk)
    dq, dk, dv = ops.attention_bwd(torch.randn_like(o), q, k, v, o, lse, causal=False, seg_q=sq, seg_k=sk)
    torch.cuda.synchronize()
    assert torch.all(o == 0) and torch.all(torch.isneginf(lse))
    assert all(torch.all(t == 0) for t in (dq, dk, dv))
    # half the keys visible: the visible half behaves like plain attention over it, nothing is NaN
    sk2 = sk.clone()
    sk2[:, :128] = 0
    o, lse = ops.attention_fwd(q, k, v, causal=False, seg_q=sq, seg_k=sk2)
    o_ref, lse_ref = ops.attention_fwd(q[:, :128].contiguous(), k[:, :128].contiguous(), v[:, :128].contiguous(), causal=False)
    torch.cuda.synchronize()
    assert not torch.isnan(o).any()
    assert _rel(o[:, :128], o_ref) < 1e-2 and _rel(lse[:, :, :128], lse_ref) < 1e-3


def test_masked_fwd_bwd_replays_in_a_cuda_graph():
    from tepdist_b200 import ops
    B, H, S = 4, 16, 1024
    qkv, q, k, v = _qkv(B, S, H, seed=4)
    do = torch.randn(B, S, H, 64, device="cuda").to(torch.bfloat16)
    seg = _layouts(B, S)["random"].cuda()

    def run():
        o, lse = ops.attention_fwd(q, k, v, causal=True, seg_q=seg, seg_k=seg)
        return (o, lse) + tuple(ops.attention_bwd(do, q, k, v, o, lse, causal=True, seg_q=seg, seg_k=seg))

    eager = [t.clone() for t in run()]       # also allocates the library's workspaces outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            outs = run()
    graph.replay()
    torch.cuda.synchronize()
    for i, (a, b) in enumerate(zip(outs, eager)):
        if i == 2:
            assert _rel(a, b) < 1e-2                 # dq: atomic order
        else:
            assert torch.equal(a, b), i


def test_gpt2_doc_mask_trains_on_one_gpu_like_the_cpu():
    import doc_mask_worker
    os.environ.pop("WORLD_SIZE", None)
    old = os.environ.get("TEPDIST_TEST_DEVICE")
    try:
        os.environ["TEPDIST_TEST_DEVICE"] = "cuda"
        gpu = doc_mask_worker.run("auto")
        os.environ["TEPDIST_TEST_DEVICE"] = "cpu"
        cpu = doc_mask_worker.run("auto")
    finally:
        if old is None:
            os.environ.pop("TEPDIST_TEST_DEVICE", None)
        else:
            os.environ["TEPDIST_TEST_DEVICE"] = old
    for a, b in zip(gpu["losses"], cpu["losses"]):
        assert abs(a - b) <= 2e-2 * max(1.0, abs(b)), (gpu, cpu)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_gpt2_doc_mask_cp2_on_two_gpus_matches_one_gpu(tmp_path):
    """n_ctx = 256: each rank's block is 128 tokens, so the ring runs the native masked kernels."""
    import doc_mask_worker
    os.environ.pop("WORLD_SIZE", None)
    env = dict(os.environ, TEPDIST_TEST_DEVICE="cuda", TEPDIST_TEST_NCTX="256")
    out = str(tmp_path / "cp2.json")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(HERE, "doc_mask_worker.py"), "cp", out]
    pr = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    assert pr.returncode == 0, pr.stderr[-3000:]
    got = json.load(open(out))["cp"]
    os.environ["TEPDIST_TEST_DEVICE"] = "cuda"
    try:
        ref = doc_mask_worker.run("auto", n_ctx=256)
    finally:
        os.environ.pop("TEPDIST_TEST_DEVICE", None)
    assert got["parallelism"] == "cp2" and got["segments_shape"] == [4, 256], got
    for a, b in zip(got["losses"], ref["losses"]):
        assert abs(a - b) <= 2e-2 * max(1.0, abs(b)), (got, ref)
