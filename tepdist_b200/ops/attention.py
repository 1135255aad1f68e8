"""Fused attention op wrappers (kernels in csrc/attention_sm100.cu).

Tensors use the "bshd" convention: q/k/v are views [B, S, H, D] (arbitrary batch/seq/head strides, D
contiguous) — typically slices of the fused qkv projection output [B, S, H, 3, D] (heads-major); the output is a
contiguous [B, S, H, D] tensor, i.e. already the [tokens, hidden] input of the output projection.

Document masking: optional int32 ids ``seg_q`` / ``seg_k`` [B, S] restrict query i to keys j with seg_q[i] == seg_k[j] (on top of
the causal rule).  Packed training windows pass the same tensor twice; a context-parallel ring block passes its query ids and
the visiting key block's ids.  A row that sees no key gets o = 0 and lse = -inf.
"""
from __future__ import annotations

import math

import torch

_HD = 64   # head dim of the tcgen05 kernels (attention_sm100.cu)


def _can_pad(S: int, D: int, causal: bool) -> bool:
    """Shapes that run on the D = 64 / S % 128 == 0 kernels through zero padding, exactly:
       * narrower heads: padded q.k terms are zero, padded V / O columns are dropped;
       * a ragged sequence length under a CAUSAL mask: padded keys sit after every real query (masked), padded query rows
         are dropped, and their zero dO makes their contribution to dK / dV vanish."""
    return D <= _HD and (S % 128 == 0 or causal)


def _pad_seg(seg_q: torch.Tensor, seg_k: torch.Tensor, S: int):
    """Pads both id tensors [B, S] to ceil128(S) with one id that no real position has (min - 1, or max + 1 when the minimum
    is INT32_MIN), so padded keys are invisible to every real query and masked calls pad exactly with or without `causal`.
    Computed on the device (no host synchronisation, capturable in a CUDA graph).  Only inputs that hold both INT32_MIN and
    INT32_MAX have no such id."""
    Sp = (S + 127) // 128 * 128
    both = torch.cat((seg_q.reshape(-1), seg_k.reshape(-1)))
    mn, mx = both.min(), both.max()
    pad = torch.where(mn > torch.iinfo(torch.int32).min, mn - 1, mx + 1)
    out = []
    for t in (seg_q, seg_k):
        o = pad.expand(t.shape[0], Sp).clone()
        o[:, :S].copy_(t)
        out.append(o)
    return out


def _visible(S: int, causal: bool, seg_q, seg_k, device):
    """Boolean [B or 1, 1, S, S] mask of the (query, key) pairs that may interact, or None for full attention."""
    mask = torch.ones(S, S, dtype=torch.bool, device=device).tril() if causal else None
    if seg_q is not None:
        m = (seg_q[:, :, None] == seg_k[:, None, :]).unsqueeze(1)
        mask = m if mask is None else m & mask
    return mask


def _pad_sd(t: torch.Tensor, S: int, D: int) -> torch.Tensor:
    """[B, S, H, D] -> zero-padded contiguous [B, ceil128(S), H, 64]."""
    Sp = (S + 127) // 128 * 128
    return torch.nn.functional.pad(t, (0, _HD - D, 0, 0, 0, Sp - S))


def _ref_fwd(q, k, v, scale, causal, seg_q=None, seg_k=None):
    # q,k,v: [B,S,H,D] -> fp32 math in [B,H,S,D]
    qf, kf, vf = (t.float().permute(0, 2, 1, 3) for t in (q, k, v))
    s = torch.matmul(qf, kf.transpose(-1, -2)) * scale
    mask = _visible(q.shape[1], causal, seg_q, seg_k, q.device)
    if mask is not None:
        s = s.masked_fill(~mask, float("-inf"))
    lse = torch.logsumexp(s, -1)  # [B,H,S]
    p = torch.exp(s - lse.unsqueeze(-1))
    if seg_q is not None:          # rows without a visible key: exp(-inf - -inf) is NaN, their probabilities are 0
        p = p.masked_fill(~mask, 0.0)
    o = torch.matmul(p, vf).permute(0, 2, 1, 3).contiguous()
    return o.to(q.dtype), lse, p


def _seg_args(seg_q, seg_k):
    if seg_q is None and seg_k is None:
        return None, None
    if seg_k is None:
        seg_k = seg_q
    if seg_q is None:
        seg_q = seg_k
    assert seg_q.shape == seg_k.shape and seg_q.dim() == 2, (seg_q.shape, seg_k.shape)
    return seg_q.to(torch.int32).contiguous(), seg_k.to(torch.int32).contiguous()


def attention_fwd(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, scale: float | None = None,
                  causal: bool = True, seg_q: torch.Tensor | None = None, seg_k: torch.Tensor | None = None):
    """Returns (o [B,S,H,D], lse [B,H,S]).  `seg_q` / `seg_k`: optional int32 document ids [B, S] (module docstring)."""
    B, S, H, D = q.shape
    if scale is None:
        scale = 1.0 / math.sqrt(D)
    seg_q, seg_k = _seg_args(seg_q, seg_k)
    if not q.is_cuda:
        o, lse, _ = _ref_fwd(q, k, v, scale, causal, seg_q, seg_k)
        return o, lse
    if D != _HD or S % 128:
        if _can_pad(S, D, causal) or (D <= _HD and seg_q is not None):
            qp, kp, vp = (_pad_sd(t, S, D) for t in (q, k, v))
            sq, sk = _pad_seg(seg_q, seg_k, S) if seg_q is not None else (None, None)
            o, lse = attention_fwd(qp, kp, vp, scale, causal, sq, sk)
            return o[:, :S, :, :D].contiguous(), lse[:, :, :S].contiguous()
        o, lse, _ = _ref_fwd(q, k, v, scale, causal, seg_q, seg_k)   # shapes the tcgen05 kernel does not cover: plain torch math
        return o, lse
    from . import lib, _check, _count, _p, _stream
    assert q.dtype == torch.bfloat16 and q.stride(3) == 1
    assert q.stride() == k.stride() == v.stride(), "q/k/v must share strides (slices of one qkv buffer)"
    o = torch.empty(B, S, H, D, dtype=q.dtype, device=q.device)
    lse = torch.empty(B, H, S, dtype=torch.float32, device=q.device)
    _check(lib().tepd_attn_fwd(q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(), lse.data_ptr(), B, H, S, D,
                               float(scale), int(causal), q.stride(0), q.stride(1), q.stride(2),
                               _p(seg_q), _p(seg_k), S, _stream()),
           "attn_fwd")
    _count(1 if seg_q is None else 2)
    return o, lse


def attention_bwd(do: torch.Tensor, q, k, v, o, lse, scale: float | None = None, causal: bool = True,
                  dqkv_out: torch.Tensor | None = None, seg_q: torch.Tensor | None = None, seg_k: torch.Tensor | None = None):
    """Returns (dq, dk, dv) as [B,S,H,D] views (of ``dqkv_out`` [B,S,H,3,D] when given).  `seg_q` / `seg_k` as in the forward."""
    B, S, H, D = q.shape
    if scale is None:
        scale = 1.0 / math.sqrt(D)
    seg_q, seg_k = _seg_args(seg_q, seg_k)
    if dqkv_out is None:
        dqkv_out = torch.empty(B, S, H, 3, D, dtype=q.dtype, device=q.device)
    dq, dk, dv = dqkv_out[:, :, :, 0], dqkv_out[:, :, :, 1], dqkv_out[:, :, :, 2]
    if q.is_cuda and (D != _HD or S % 128) and (_can_pad(S, D, causal) or (D <= _HD and seg_q is not None)):
        Sp = (S + 127) // 128 * 128
        lse_p = lse if Sp == S else torch.nn.functional.pad(lse, (0, Sp - S))
        sq, sk = _pad_seg(seg_q, seg_k, S) if seg_q is not None else (None, None)
        gq, gk, gv = attention_bwd(_pad_sd(do, S, D), _pad_sd(q, S, D), _pad_sd(k, S, D), _pad_sd(v, S, D), _pad_sd(o, S, D),
                                   lse_p, scale, causal, seg_q=sq, seg_k=sk)
        dq.copy_(gq[:, :S, :, :D]); dk.copy_(gk[:, :S, :, :D]); dv.copy_(gv[:, :S, :, :D])
        return dq, dk, dv
    if not q.is_cuda or D != _HD or S % 128:
        dof = do.float().permute(0, 2, 1, 3)
        qf, kf, vf = (t.float().permute(0, 2, 1, 3) for t in (q, k, v))
        # probabilities from the GIVEN log-sum-exp (like the kernels): a block of a longer key sequence (ring attention) passes
        # the log-sum-exp over ALL keys, and its probabilities must not be re-normalised over the block
        sc = torch.matmul(qf, kf.transpose(-1, -2)) * scale
        mask = _visible(S, causal, seg_q, seg_k, q.device)
        if mask is not None:
            sc = sc.masked_fill(~mask, float("-inf"))
        p = torch.exp(sc - lse.float().unsqueeze(-1))
        if seg_q is not None:      # rows with lse = -inf (no visible key): exact zeros, not NaN
            p = p.masked_fill(~mask, 0.0)
        dvf = torch.matmul(p.transpose(-1, -2), dof)
        dp = torch.matmul(dof, vf.transpose(-1, -2))
        delta = (dof * o.float().permute(0, 2, 1, 3)).sum(-1, keepdim=True)
        ds = p * (dp - delta) * scale
        dqf = torch.matmul(ds, kf)
        dkf = torch.matmul(ds.transpose(-1, -2), qf)
        dq.copy_(dqf.permute(0, 2, 1, 3).to(q.dtype))
        dk.copy_(dkf.permute(0, 2, 1, 3).to(q.dtype))
        dv.copy_(dvf.permute(0, 2, 1, 3).to(q.dtype))
        return dq, dk, dv
    from . import lib, _check, _count, _p, _stream
    do = do.contiguous()
    assert o.is_contiguous() and do.is_contiguous()
    # dq accumulator: persistent self-clearing fp32 workspace inside the library (no per-call memset)
    _check(lib().tepd_attn_bwd(do.data_ptr(), q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(), lse.data_ptr(),
                               None, dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), B, H, S, D,
                               float(scale), int(causal), q.stride(0), q.stride(1), q.stride(2),
                               dq.stride(0), dq.stride(1), dq.stride(2), _p(seg_q), _p(seg_k), S, _stream()), "attn_bwd")
    _count(3 if seg_q is None else 4)
    return dq, dk, dv


# --------------------------------------------------------------------------------------------- ring (context-parallel) helpers
def _native_ring(*ts: torch.Tensor) -> bool:
    return all(t.is_cuda and t.is_contiguous() for t in ts) and ts[0].shape[-1] % 8 == 0


def attn_merge_(o_acc: torch.Tensor, lse_acc: torch.Tensor, lse_out: torch.Tensor, o_j: torch.Tensor, lse_j: torch.Tensor,
                first: bool) -> torch.Tensor:
    """Log-sum-exp merge of one block's partial attention (o_j [B,L,H,D], lse_j [B,H,L]) into the running fp32 pair
    (o_acc in place; the merged log-sum-exp goes to `lse_out`, which is returned).  One kernel (elementwise_sm100.cu
    attn_merge_kernel); plain torch math on CPU."""
    B, L, H, D = o_j.shape
    if o_j.dtype == torch.bfloat16 and _native_ring(o_j, o_acc, lse_acc, lse_out, lse_j):
        from . import lib, _check, _count, _stream
        _check(lib().tepd_attn_merge(o_acc.data_ptr(), lse_acc.data_ptr(), lse_out.data_ptr(), o_j.data_ptr(), lse_j.data_ptr(),
                                     B, L, H, D, int(first), _stream()), "attn_merge")
        _count()
        return lse_out
    if first:
        o_acc.copy_(o_j)
        lse_out.copy_(lse_j)
        return lse_out
    new = torch.logaddexp(lse_acc, lse_j)
    empty = torch.isneginf(new)        # no visible key in either partial (document masking): stay at o = 0, lse = -inf
    wa = torch.exp(lse_acc - new).masked_fill(empty, 0.0).permute(0, 2, 1).unsqueeze(-1)     # [B,L,H,1]
    wj = torch.exp(lse_j - new).masked_fill(empty, 0.0).permute(0, 2, 1).unsqueeze(-1)
    o_acc.mul_(wa).add_(o_j.float() * wj)
    lse_out.copy_(new)
    return lse_out


def attn_ring_accum_(dq_acc: torch.Tensor, kv_acc: torch.Tensor, part: torch.Tensor) -> None:
    """dq_acc [B,L,H,D] += part[..,0,:]; kv_acc [B,L,H,2,D] += part[..,1:,:] (part [B,L,H,3,D]: one block's dq / dk / dv)."""
    if part.dtype == torch.bfloat16 and _native_ring(part, dq_acc, kv_acc):
        from . import lib, _check, _count, _stream
        _check(lib().tepd_attn_ring_accum(dq_acc.data_ptr(), kv_acc.data_ptr(), part.data_ptr(), dq_acc.numel() // dq_acc.shape[-1],
                                          dq_acc.shape[-1], 0, _stream()), "attn_ring_accum")
        _count()
        return
    dq_acc += part[:, :, :, 0]
    kv_acc += part[:, :, :, 1:]


def attn_ring_pack(dq_acc: torch.Tensor, kv_acc: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """out [B,L,H,3,D] (compute dtype) <- the fp32 accumulators at the end of the ring."""
    if out.dtype == torch.bfloat16 and _native_ring(out, dq_acc, kv_acc):
        from . import lib, _check, _count, _stream
        _check(lib().tepd_attn_ring_accum(dq_acc.data_ptr(), kv_acc.data_ptr(), out.data_ptr(), dq_acc.numel() // dq_acc.shape[-1],
                                          dq_acc.shape[-1], 1, _stream()), "attn_ring_pack")
        _count()
        return out
    out[:, :, :, 0].copy_(dq_acc)
    out[:, :, :, 1:].copy_(kv_acc)
    return out
