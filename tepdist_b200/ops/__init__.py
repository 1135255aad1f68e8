"""Device-op layer: hand-written sm_100a kernels behind a C ABI (``libtepdist_kernels.so``), loaded with
ctypes.  On CUDA tensors every op here runs OUR kernel and raises if the library is missing (no silent
eager fallback); CPU tensors take a plain-PyTorch reference path that the tests also use as the oracle.

Launch accounting: ``launch_count()`` returns how many of our kernels were launched (bench.py reports it
as ``gpu_launches``).
"""
from __future__ import annotations

import ctypes
import math
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libtepdist_kernels.so")
_lib: Optional[ctypes.CDLL] = None
_launches = 0
_num_sms: Optional[int] = None


class KernelLibraryMissing(RuntimeError):
    pass


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise KernelLibraryMissing(
                f"{_LIB_PATH} not built; run `python -m tepdist_b200.build_native` (nvcc, sm_100a)")
        _lib = ctypes.CDLL(_LIB_PATH)
        for name in dir(_Sig):
            if name.startswith("tepd_"):
                try:
                    fn = getattr(_lib, name)
                except AttributeError:  # symbol not in this build
                    continue
                fn.restype = ctypes.c_int
                fn.argtypes = getattr(_Sig, name)
    return _lib


def available() -> bool:
    return os.path.exists(_LIB_PATH)


def launch_count() -> int:
    return _launches


def reset_launch_count() -> None:
    global _launches
    _launches = 0


_warned: set = set()


def _warn_once(msg: str) -> None:
    if msg not in _warned:
        _warned.add(msg)
        import warnings
        warnings.warn(msg)


def _count(n: int = 1) -> None:
    global _launches
    _launches += n


_vp, _i, _ll, _f = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_float


class _Sig:
    tepd_gemm_bf16 = [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _ll, _ll, _ll, _ll, _ll, _ll, _ll, _ll,
                      _i, _i, _i, _i, _i, _i, _f, _i, _i, _i, _vp, _vp, _vp]
    tepd_gemm2_bf16 = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _ll, _ll, _ll, _ll, _i, _i, _i, _f, _i, _vp, _i, _i, _i]
    tepd_layernorm_fwd = [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _vp]
    tepd_layernorm_bwd = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp]
    tepd_gelu_fwd = [_vp, _vp, _ll, _vp]
    tepd_gelu_bwd = [_vp, _vp, _vp, _ll, _vp]
    tepd_colsum = [_vp, _vp, _i, _i, _vp]
    tepd_bn_fwd_nhwc = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _i, _vp]
    tepd_bn_bwd_nhwc = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp]
    tepd_bn_reduce_nhwc = [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]
    tepd_bn_fwd_apply_nhwc = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _i, _f, _vp]
    tepd_bn_bwd_apply_nhwc = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _vp]
    tepd_im2col_nhwc = [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]
    tepd_col2im_nhwc = [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]
    tepd_embedding_fwd = [_vp, _vp, _vp, _vp, _i, _i, _i, _vp]
    tepd_embedding_bwd = [_vp, _vp, _vp, _vp, _i, _i, _i, _vp]
    tepd_xent_fwd_bwd = [_vp, _vp, _vp, _vp, _i, _i, _i, _f, _vp]
    tepd_adamw = [_vp, _vp, _vp, _vp, _vp, _ll, _ll, _f, _f, _f, _f, _f, _f, _f, _f, _vp, _vp]
    tepd_sgd = [_vp, _vp, _vp, _ll, _f, _f, _vp]
    tepd_axpy_f32 = [_vp, _vp, _ll, _f, _vp]
    tepd_cast_f32_bf16 = [_vp, _vp, _ll, _vp]
    tepd_ew_bf16 = [_vp, _vp, _vp, _ll, _i, _vp]
    tepd_moe_gather_scale = [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]
    tepd_moe_combine_sum = [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]
    tepd_moe_route_dots = [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]
    tepd_maxpool_nhwc = [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]
    tepd_maxpool_bwd_nhwc = [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]
    tepd_gap_nhwc = [_vp, _vp, _i, _i, _i, _vp]
    tepd_gap_bwd_nhwc = [_vp, _vp, _i, _i, _i, _vp]
    tepd_attn_merge = [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]
    tepd_attn_ring_accum = [_vp, _vp, _vp, _ll, _i, _i, _vp]
    tepd_attn_fwd = [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, _i, _ll, _ll, _ll, _vp, _vp, _ll, _vp]
    tepd_attn_bwd = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, _i,
                     _ll, _ll, _ll, _ll, _ll, _ll, _vp, _vp, _ll, _vp]


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _sms() -> int:
    global _num_sms
    if _num_sms is None:
        _num_sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    return _num_sms


def _check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"tepdist_b200 kernel '{what}' failed with code {rc}")


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


# --------------------------------------------------------------------------------------------- GEMM
def gemm(a: torch.Tensor, b: torch.Tensor, *, a_mn: bool = False, b_mn: bool = False,
         bias: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None,
         act: Optional[str] = None, out: Optional[torch.Tensor] = None,
         out_dtype: torch.dtype = torch.bfloat16, accumulate: bool = False, alpha: float = 1.0,
         split_k: int = 0, block_n: int = 0, out2: Optional[torch.Tensor] = None,
         aux: Optional[torch.Tensor] = None) -> torch.Tensor:
    """D = act(alpha * A @ B + bias) + residual with A:(M,K), B:(K,N) as *logical* shapes.

    Storage: ``a`` is [.., M, K] (a_mn=False) or [.., K, M] (a_mn=True); ``b`` is [.., N, K]
    (b_mn=False, i.e. nn.Linear weight layout) or [.., K, N] (b_mn=True).  Optional leading batch dim.
    ``accumulate`` adds into an fp32 ``out`` (gradient accumulation / split-K reduction target).
    ``act="gelu"`` with ``out2``: ``out`` receives the pre-activation, ``out2`` the activated value (one pass).
    ``act="gelu_bwd"`` with ``aux`` (pre-activation): the result is multiplied by GELU'(aux) in the epilogue.
    """
    assert a.dim() == b.dim() and a.dim() in (2, 3)
    batched = a.dim() == 3
    if not batched:
        a3, b3 = a.unsqueeze(0), b.unsqueeze(0)
    else:
        a3, b3 = a, b
    batch = a3.shape[0]
    M, K = (a3.shape[2], a3.shape[1]) if a_mn else (a3.shape[1], a3.shape[2])
    N, Kb = (b3.shape[2], b3.shape[1]) if b_mn else (b3.shape[1], b3.shape[2])
    assert K == Kb, f"contraction mismatch {K} vs {Kb}"
    if out is None:
        shape = (batch, M, N) if batched else (M, N)
        out = torch.empty(shape, dtype=out_dtype, device=a.device)
        assert not accumulate
    out3 = out.unsqueeze(0) if out.dim() == 2 else out

    odd = a.is_cuda and (N % 8 != 0 or (a_mn and M % 8 != 0) or (K % 8 != 0 and not (a_mn and b_mn))
                         or a.dtype != torch.bfloat16 or b.dtype != torch.bfloat16)
    if odd:
        _warn_once(f"gemm {M}x{N}x{K} ({a.dtype}): shape / dtype outside the TMA alignment rules of the tcgen05 kernels, "
                   "running this one through torch.matmul")
    if not a.is_cuda or odd:  # reference path (CPU tests / oracle; odd shapes on the GPU)
        A = a3.float().transpose(1, 2) if a_mn else a3.float()
        B = b3.float() if b_mn else b3.float().transpose(1, 2)
        d = alpha * torch.matmul(A, B)
        if bias is not None:
            d = d + bias.float()
        if act == "gelu":
            if out2 is not None:
                out2.reshape(d.shape).copy_(torch.nn.functional.gelu(d, approximate="tanh").to(out2.dtype))
            else:
                d = torch.nn.functional.gelu(d, approximate="tanh")
        if act == "gelu_bwd":
            xa = aux.float().reshape(d.shape).detach().requires_grad_(True)
            with torch.enable_grad():
                ya = torch.nn.functional.gelu(xa, approximate="tanh")
            (ga,) = torch.autograd.grad(ya, xa, torch.ones_like(ya))
            d = d * ga
        if residual is not None:
            d = d + residual.float().reshape(d.shape)
        if accumulate:
            out3.add_(d.to(out.dtype))
        else:
            out3.copy_(d.to(out.dtype))
        return out

    assert a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16
    assert a3.stride(2) == 1 and b3.stride(2) == 1 and out3.stride(2) == 1
    if STREAM_K_FWD and split_k == 0 and block_n == 0 and not batched and not accumulate and K >= 512:
        # wave quantisation check for the persistent 128x256 schedule: below ~93 % SM occupancy the stream-K schedule
        # (equal k-block ranges per SM + workspace fix-up of split tiles) wins over both tile-parallel kernels
        tiles = ((M + 127) // 128) * ((N + 255) // 256)
        waves = -(-tiles // _sms())
        if tiles / (waves * _sms()) < 0.93:
            split_k = -1
    if (USE_GEMM2 and not batched and not a_mn and not accumulate and out.dtype == torch.bfloat16 and M >= 256 and N >= 256
            and block_n == 0 and split_k in (0, 1)):
        res2 = None if residual is None else residual.reshape(M, N)
        gemm2(a, b, b_mn=b_mn, bias=bias, residual=res2, act=act, out=out, out2=out2,
              aux=None if aux is None else aux.reshape(M, N), alpha=alpha)
        return out
    if (USE_GEMM2 and not batched and a_mn and b_mn and not accumulate and out.dtype == torch.float32 and M >= 256 and N >= 256
            and block_n == 0 and split_k in (0, 1) and bias is None and residual is None and act is None):
        gemm2(a, b, a_mn=True, b_mn=True, out=out, alpha=alpha)     # weight gradient with plain stores
        return out
    if bias is not None:
        assert bias.dtype in (torch.float32, torch.bfloat16) and bias.is_contiguous()
    res3 = None
    if residual is not None:
        res3 = residual.reshape(out3.shape)
        assert res3.dtype == torch.bfloat16 and res3.stride(2) == 1
    if split_k == 0:
        split_k = 1
        if accumulate and out.dtype == torch.float32:
            tiles = ((M + 127) // 128) * ((N + 255) // 256) * batch
            kb = (K + 63) // 64
            if STREAM_K and tiles >= _sms():
                split_k = -1    # stream-K: every SM gets the same number of k-blocks (fp32 red.add flush per tile); measured
                                # neutral-to-better from one full wave of tiles up, worse than plain split-K below that
            else:
                while tiles * split_k * 2 <= _sms() and split_k * 2 <= max(1, kb // 4):
                    split_k *= 2
    rc = lib().tepd_gemm_bf16(
        a3.data_ptr(), b3.data_ptr(), out3.data_ptr(), _p(bias), _p(res3),
        M, N, K, batch, a3.stride(1), b3.stride(1), out3.stride(1),
        a3.stride(0), b3.stride(0), out3.stride(0),
        res3.stride(1) if res3 is not None else 0, res3.stride(0) if res3 is not None else 0,
        int(a_mn), int(b_mn), int(out.dtype == torch.float32), int(accumulate),
        {None: 0, "gelu": 1, "gelu_bwd": 2}[act], int(bias is not None and bias.dtype == torch.bfloat16),
        float(alpha), int(split_k), int(block_n), _sms(), _stream(), _p(out2),
        _p(aux.reshape(out3.shape) if aux is not None else None))
    _check(rc, "gemm_bf16")
    _count()
    return out


STREAM_K_FWD = os.environ.get("TEPDIST_STREAM_K_FWD", "0") == "1"   # stream-K + fix-up for bf16-output GEMMs (opt-in)
STREAM_K = os.environ.get("TEPDIST_STREAM_K", "1") == "1"  # stream-K scheduling for fp32-accumulate GEMMs (weight gradients)
USE_GEMM2 = os.environ.get("TEPDIST_GEMM2", "1") == "1"   # 2-CTA (cta_group::2) kernel for eligible shapes (measured +1.7 % on the GPT-2 step)


def wgrad_prefers_store(n_out: int, k_in: int) -> bool:
    """Weight gradient [n_out, k_in]: plain-store 2-CTA GEMM when the 256x256 tiles fill at least half of the CTA pairs;
    smaller outputs are better off split over K with fp32 red.add into a zero-filled slot (1-CTA kernel)."""
    tiles = ((n_out + 255) // 256) * ((k_in + 255) // 256)
    return USE_GEMM2 and n_out >= 256 and k_in >= 256 and n_out % 8 == 0 and k_in % 8 == 0 and tiles * 2 >= _sms() // 2


def _gemm2_stream_k(M: int, N: int, K: int, fp32_out: bool) -> bool:
    """Measured (profiles/kernel_checks_trip22.json): the stream-K schedule of the 2-CTA kernel only pays for very large
    plain-store outputs (lm_head weight gradient 50304x1024: 1466 vs 1245 TFLOP/s); on the 64..256-tile transformer shapes
    the fix-up of split tiles (uncoalesced fp32 partial tiles through L2) costs more than the idle tail wave it removes."""
    if not STREAM_K or not fp32_out:
        return False
    tiles = ((M + 255) // 256) * ((N + 255) // 256)
    return tiles >= 8 * (_sms() // 2)


def gemm2(a: torch.Tensor, b: torch.Tensor, *, a_mn: bool = False, b_mn: bool = False, bias: Optional[torch.Tensor] = None,
          residual: Optional[torch.Tensor] = None, act: Optional[str] = None, out: Optional[torch.Tensor] = None,
          out2: Optional[torch.Tensor] = None, aux: Optional[torch.Tensor] = None, alpha: float = 1.0,
          out_dtype: torch.dtype = torch.bfloat16, stream_k: Optional[bool] = None) -> torch.Tensor:
    """2-CTA tcgen05 GEMM (256x256 tile per CTA pair): a [M,K] (or [K,M] with a_mn), b [N,K] (or [K,N] with b_mn);
    bf16 output with the fused epilogues or fp32 plain stores.  stream_k: None = decide from the wave occupancy."""
    M, K = (a.shape[1], a.shape[0]) if a_mn else a.shape
    N = b.shape[1] if b_mn else b.shape[0]
    if out is None:
        out = torch.empty(M, N, dtype=out_dtype, device=a.device)
    assert a.is_cuda and a.dtype == torch.bfloat16 and a.stride(1) == 1 and b.stride(1) == 1 and out.stride(1) == 1
    assert out.dtype in (torch.bfloat16, torch.float32)
    if stream_k is None:
        stream_k = _gemm2_stream_k(M, N, K, out.dtype == torch.float32)
    rc = lib().tepd_gemm2_bf16(a.data_ptr(), b.data_ptr(), out.data_ptr(), _p(out2), _p(bias), _p(residual), _p(aux), M, N, K,
                               a.stride(0), b.stride(0), out.stride(0), residual.stride(0) if residual is not None else 0,
                               int(b_mn), {None: 0, "gelu": 1, "gelu_bwd": 2}[act],
                               int(bias is not None and bias.dtype == torch.bfloat16), float(alpha), _sms(), _stream(),
                               int(a_mn), int(out.dtype == torch.float32), int(bool(stream_k)))
    _check(rc, "gemm2_bf16")
    _count()
    return out


def einsum(eq: str, a: torch.Tensor, b: torch.Tensor, _force: bool = False) -> torch.Tensor:
    """Two-operand einsum as ONE batched tcgen05 GEMM (the expert FFNs / dispatch / combine of GPT-MoE and their gradients are
    einsums with a leading expert or group dim; the reference hands them to cuBLAS batched GEMMs, SURVEY 2.H K8).

    Indices are classified batch (in a, b, out) / M (a, out) / N (b, out) / K (a, b): each operand is brought to
    [batch, rows, cols] with its groups kept in memory order when they already are (either major is fine: the kernel reads
    K-major and MN-major operands alike through TMA), copied once otherwise; the [batch, M, N] result is viewed / permuted
    to the requested output order.  Falls back to torch.einsum for index patterns or shapes outside the kernel's alignment
    rules (dims % 8, bf16)."""
    lhs, out_idx = eq.replace(" ", "").split("->")
    ia, ib = lhs.split(",")
    ok = (((a.is_cuda and a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16) or _force) and len(set(ia)) == len(ia)
          and len(set(ib)) == len(ib) and len(set(out_idx)) == len(out_idx))
    if ok:
        batch = [c for c in out_idx if c in ia and c in ib]
        m_idx = [c for c in ia if c in out_idx and c not in ib]
        n_idx = [c for c in ib if c in out_idx and c not in ia]
        k_idx = [c for c in ia if c in ib and c not in out_idx]
        ok = (len(batch) + len(m_idx) + len(k_idx) == len(ia) and len(batch) + len(n_idx) + len(k_idx) == len(ib)
              and bool(m_idx) and bool(n_idx) and bool(k_idx))
    if not ok:
        return torch.einsum(eq, a, b)
    size = {c: d for c, d in zip(ia, a.shape)}
    size.update({c: d for c, d in zip(ib, b.shape)})
    prod = lambda idx: int(math.prod(size[c] for c in idx)) if idx else 1
    B_, M, N, K = prod(batch), prod(m_idx), prod(n_idx), prod(k_idx)
    if M % 8 or N % 8 or K % 8:
        return torch.einsum(eq, a, b)

    def arrange(t: torch.Tensor, idx: str, rows, cols):
        """-> (tensor [B, R, C] contiguous, transposed?) choosing rows-major or cols-major storage, whichever needs no copy."""
        for first, second, tr in ((rows, cols, False), (cols, rows, True)):
            want = "".join(batch + first + second)
            if want == idx and t.is_contiguous():
                return t.reshape(B_, prod(first), prod(second)), tr
        perm = [idx.index(c) for c in batch + rows + cols]
        return t.permute(perm).contiguous().reshape(B_, prod(rows), prod(cols)), False

    a3, a_tr = arrange(a, ia, m_idx, k_idx)        # [B, M, K] or (a_tr) [B, K, M]
    b3, b_tr = arrange(b, ib, k_idx, n_idx)        # [B, K, N] or (b_tr) [B, N, K]
    if B_ == 1:
        d = gemm(a3[0], b3[0], a_mn=a_tr, b_mn=not b_tr).unsqueeze(0)
    else:
        d = gemm(a3, b3, a_mn=a_tr, b_mn=not b_tr)
    d = d.reshape([size[c] for c in batch + m_idx + n_idx])
    cur = "".join(batch + m_idx + n_idx)
    if cur != out_idx:
        d = d.permute([cur.index(c) for c in out_idx]).contiguous()
    return d


def _dense_same_layout(*ts: torch.Tensor) -> bool:
    """All tensors bf16 on the GPU, same shape and strides, dense in memory (any of contiguous / channels_last): an elementwise
    kernel may then walk the raw storage linearly."""
    t0 = ts[0]
    if not (t0.is_cuda and t0.dtype == torch.bfloat16 and t0.numel() % 8 == 0 and t0.numel() > 0):
        return False
    if not (t0.is_contiguous() or (t0.dim() == 4 and t0.is_contiguous(memory_format=torch.channels_last))):
        return False
    return all(t.dtype == t0.dtype and t.shape == t0.shape and t.stride() == t0.stride() and t.is_cuda for t in ts[1:])


def ew_native(mode: str, a: torch.Tensor, b: Optional[torch.Tensor] = None) -> Optional[torch.Tensor]:
    """relu(a) | relu_bwd: a * (b > 0) | add: a + b with the own vectorised kernel; None when the operands do not qualify
    (the caller then uses the torch op)."""
    ts = (a,) if b is None else (a, b)
    if not _dense_same_layout(*ts):
        return None
    out = torch.empty_like(a)
    rc = lib().tepd_ew_bf16(a.data_ptr(), a.data_ptr() if b is None else b.data_ptr(), out.data_ptr(), a.numel(),
                            {"relu": 0, "relu_bwd": 1, "add": 2}[mode], _stream())
    _check(rc, "ew_bf16")
    _count()
    return out


# --------------------------------------------------------------------------------------------- MoE route-table kernels
def moe_gather_scale(src: torch.Tensor, slot_src: torch.Tensor, w: torch.Tensor, E: int, C: int) -> torch.Tensor:
    """out[e, g, c, :] = w[g, e, c] * src[g, slot_src[g, e, c], :] (zero where slot_src < 0).  src [G, S, M]; slot_src int32 [G, E, C]."""
    G, S, M = src.shape
    if not src.is_cuda or src.dtype != torch.bfloat16 or M % 8:
        valid = slot_src >= 0
        idx = slot_src.clamp(min=0).long().reshape(G, E * C)
        rows = torch.gather(src.float(), 1, idx.unsqueeze(-1).expand(G, E * C, M)).reshape(G, E, C, M)
        out = rows * (w.float() * valid).unsqueeze(-1)
        return out.permute(1, 0, 2, 3).contiguous().to(src.dtype)
    out = torch.empty(E, G, C, M, dtype=src.dtype, device=src.device)
    _check(lib().tepd_moe_gather_scale(src.contiguous().data_ptr(), slot_src.contiguous().data_ptr(), w.contiguous().data_ptr(),
                                       out.data_ptr(), G, S, E, C, M, _stream()), "moe_gather_scale")
    _count()
    return out


def moe_combine_sum(y: torch.Tensor, re: torch.Tensor, rc: torch.Tensor, gw: torch.Tensor, S: int) -> torch.Tensor:
    """out[g, s, :] = sum_k gw[g, s, k] * y[re[g, s, k], g, rc[g, s, k], :] (routes with re < 0 dropped).  y [E, G, C, M]."""
    E, G, C, M = y.shape
    K = re.shape[-1]
    if not y.is_cuda or y.dtype != torch.bfloat16 or M % 8:
        yg = y.float().permute(1, 0, 2, 3).reshape(G, E * C, M)
        flat = (re.clamp(min=0).long() * C + rc.clamp(min=0).long()).reshape(G, S * K)
        rows = torch.gather(yg, 1, flat.unsqueeze(-1).expand(G, S * K, M)).reshape(G, S, K, M)
        out = (rows * (gw.float() * (re >= 0)).unsqueeze(-1)).sum(2)
        return out.to(y.dtype)
    out = torch.empty(G, S, M, dtype=y.dtype, device=y.device)
    _check(lib().tepd_moe_combine_sum(y.contiguous().data_ptr(), re.contiguous().data_ptr(), rc.contiguous().data_ptr(),
                                      gw.contiguous().data_ptr(), out.data_ptr(), G, S, E, C, M, K, _stream()), "moe_combine_sum")
    _count()
    return out


def moe_route_dots(a: torch.Tensor, b: torch.Tensor, re: torch.Tensor, rc: torch.Tensor) -> torch.Tensor:
    """dots[g, s, k] = < a[g, s, :], b[re[g, s, k], g, rc[g, s, k], :] > (0 for dropped routes), fp32.  a [G, S, M]; b [E, G, C, M]."""
    G, S, M = a.shape
    E, _, C, _ = b.shape
    K = re.shape[-1]
    if not a.is_cuda or a.dtype != torch.bfloat16 or M % 8:
        bg = b.float().permute(1, 0, 2, 3).reshape(G, E * C, M)
        flat = (re.clamp(min=0).long() * C + rc.clamp(min=0).long()).reshape(G, S * K)
        rows = torch.gather(bg, 1, flat.unsqueeze(-1).expand(G, S * K, M)).reshape(G, S, K, M)
        return ((rows * a.float().unsqueeze(2)).sum(-1) * (re >= 0)).float()
    dots = torch.empty(G, S, K, dtype=torch.float32, device=a.device)
    _check(lib().tepd_moe_route_dots(a.contiguous().data_ptr(), b.contiguous().data_ptr(), re.contiguous().data_ptr(),
                                     rc.contiguous().data_ptr(), dots.data_ptr(), G, S, E, C, M, K, _stream()), "moe_route_dots")
    _count()
    return dots


# --------------------------------------------------------------------------------------------- convolution
CONV_NATIVE = os.environ.get("TEPDIST_CONV", "native") != "cudnn"   # "cudnn": library path (the reference's K9)


def conv_native_ok(x: torch.Tensor, w: torch.Tensor) -> bool:
    """Own path: NHWC im2col / col2im kernels (conv_sm100.cu) around the tcgen05 GEMMs."""
    return CONV_NATIVE and x.is_cuda and x.dtype == torch.bfloat16 and w.shape[0] % 8 == 0


def _conv_geom(x_shape, w_shape, stride: int, pad: int):
    N, C, H, W = x_shape
    Cout, Cin, kh, kw = w_shape
    Ho, Wo = (H + 2 * pad - kh) // stride + 1, (W + 2 * pad - kw) // stride + 1
    Kpad = (kh * kw * C + 7) // 8 * 8
    direct = kh == 1 and kw == 1 and stride == 1 and pad == 0 and C % 8 == 0     # the convolution IS a GEMM
    return N, C, H, W, Cout, kh, kw, Ho, Wo, Kpad, direct


def _nhwc(x: torch.Tensor) -> torch.Tensor:
    """[N, C, H, W] (any strides) -> contiguous [N, H, W, C] view of channels_last memory."""
    return x.contiguous(memory_format=torch.channels_last).permute(0, 2, 3, 1)


def _conv_weight_matrix(w: torch.Tensor, Kpad: int) -> torch.Tensor:
    """OIHW -> [Cout, (tap, cin)] bf16, K padded with zeros (tap-major columns match im2col)."""
    Cout = w.shape[0]
    m = w.permute(0, 2, 3, 1).reshape(Cout, -1).to(torch.bfloat16)
    if m.shape[1] != Kpad:
        m = torch.nn.functional.pad(m, (0, Kpad - m.shape[1]))
    return m.contiguous()


def _im2col(xn: torch.Tensor, g) -> torch.Tensor:
    N, C, H, W, Cout, kh, kw, Ho, Wo, Kpad, direct = g
    if direct:
        return xn.reshape(N * H * W, C)
    col = torch.empty(N * Ho * Wo, Kpad, dtype=torch.bfloat16, device=xn.device)
    return col


def conv2d_fwd(x: torch.Tensor, w: torch.Tensor, stride: int, pad: int) -> torch.Tensor:
    """x [N,C,H,W] bf16, w [Cout,Cin,kh,kw] -> y [N,Cout,Ho,Wo] (channels_last memory)."""
    g = _conv_geom(x.shape, w.shape, stride, pad)
    N, C, H, W, Cout, kh, kw, Ho, Wo, Kpad, direct = g
    xn = _nhwc(x)
    col = _im2col(xn, g)
    if not direct:
        _check(lib().tepd_im2col_nhwc(xn.data_ptr(), col.data_ptr(), N, H, W, C, Ho, Wo, kh, kw, stride, pad, Kpad, _stream()), "im2col")
        _count()
    y = gemm(col, _conv_weight_matrix(w, Kpad))
    return y.view(N, Ho, Wo, Cout).permute(0, 3, 1, 2)


def conv2d_dgrad(dy: torch.Tensor, w: torch.Tensor, x_shape, stride: int, pad: int) -> torch.Tensor:
    g = _conv_geom(x_shape, w.shape, stride, pad)
    N, C, H, W, Cout, kh, kw, Ho, Wo, Kpad, direct = g
    dyn = _nhwc(dy).reshape(N * Ho * Wo, Cout)
    dcol = gemm(dyn, _conv_weight_matrix(w, Kpad), b_mn=True)            # [rows, Kpad]
    if direct:
        return dcol.view(N, H, W, C).permute(0, 3, 1, 2)
    dx = torch.empty(N, H, W, C, dtype=torch.bfloat16, device=dy.device)
    _check(lib().tepd_col2im_nhwc(dcol.data_ptr(), dx.data_ptr(), N, H, W, C, Ho, Wo, kh, kw, stride, pad, Kpad, _stream()), "col2im")
    _count()
    return dx.permute(0, 3, 1, 2)


def conv2d_wgrad(dy: torch.Tensor, x: torch.Tensor, w_shape, stride: int, pad: int) -> torch.Tensor:
    """fp32 [Cout, Cin, kh, kw] = dY^T . im2col(x)."""
    g = _conv_geom(x.shape, w_shape, stride, pad)
    N, C, H, W, Cout, kh, kw, Ho, Wo, Kpad, direct = g
    xn = _nhwc(x)
    col = _im2col(xn, g)
    if not direct:
        _check(lib().tepd_im2col_nhwc(xn.data_ptr(), col.data_ptr(), N, H, W, C, Ho, Wo, kh, kw, stride, pad, Kpad, _stream()), "im2col")
        _count()
    dyn = _nhwc(dy).reshape(N * Ho * Wo, Cout)
    gw = gemm(dyn, col, a_mn=True, b_mn=True, out_dtype=torch.float32)   # [Cout, Kpad]
    return gw[:, :kh * kw * C].reshape(Cout, kh, kw, C).permute(0, 3, 1, 2)


# --------------------------------------------------------------------------------------------- pooling (NHWC kernels, conv_sm100.cu)
def pool_native_ok(x: torch.Tensor) -> bool:
    return CONV_NATIVE and x.is_cuda and x.dtype == torch.bfloat16 and x.dim() == 4 and x.shape[1] % 8 == 0 and x.numel() > 0


def _cl(x: torch.Tensor) -> torch.Tensor:
    return x.contiguous(memory_format=torch.channels_last)


def maxpool2d_fwd(x: torch.Tensor, k: int, stride: int, pad: int) -> torch.Tensor:
    """[N, C, H, W] -> [N, C, Ho, Wo] (floor mode, -inf padding); own kernel on channels_last bf16, torch elsewhere."""
    if not pool_native_ok(x):
        return torch.nn.functional.max_pool2d(x, k, stride, pad)
    N, C, H, W = x.shape
    Ho, Wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    xc = _cl(x)
    y = torch.empty((N, C, Ho, Wo), dtype=x.dtype, device=x.device, memory_format=torch.channels_last)
    _check(lib().tepd_maxpool_nhwc(xc.data_ptr(), y.data_ptr(), N, H, W, C, Ho, Wo, k, stride, pad, _stream()), "maxpool")
    _count()
    return y


def maxpool2d_bwd(dy: torch.Tensor, x: torch.Tensor, y: torch.Tensor, k: int, stride: int, pad: int) -> torch.Tensor:
    """Gradient of max_pool2d given the forward input and output (gather form, first-maximum tie rule like torch)."""
    if not (pool_native_ok(x) and dy.dtype == x.dtype and y.dtype == x.dtype):
        xr = x.detach().float().requires_grad_(True)
        with torch.enable_grad():
            yy = torch.nn.functional.max_pool2d(xr, k, stride, pad)
        (gx,) = torch.autograd.grad(yy, xr, dy.float())
        return gx.to(x.dtype)
    N, C, H, W = x.shape
    Ho, Wo = y.shape[2], y.shape[3]
    dx = torch.empty((N, C, H, W), dtype=x.dtype, device=x.device, memory_format=torch.channels_last)
    _check(lib().tepd_maxpool_bwd_nhwc(_cl(dy).data_ptr(), _cl(x).data_ptr(), _cl(y).data_ptr(), dx.data_ptr(), N, H, W, C, Ho, Wo, k, stride,
                                       pad, _stream()), "maxpool_bwd")
    _count()
    return dx


def global_avgpool_fwd(x: torch.Tensor) -> torch.Tensor:
    if not pool_native_ok(x):
        return x.float().mean((2, 3)).to(x.dtype)
    N, C, H, W = x.shape
    y = torch.empty(N, C, dtype=x.dtype, device=x.device)
    _check(lib().tepd_gap_nhwc(_cl(x).data_ptr(), y.data_ptr(), N, H * W, C, _stream()), "gap")
    _count()
    return y


def global_avgpool_bwd(dy: torch.Tensor, shape) -> torch.Tensor:
    N, C, H, W = shape
    if not (CONV_NATIVE and dy.is_cuda and dy.dtype == torch.bfloat16 and C % 8 == 0):
        return (dy / (H * W)).view(N, C, 1, 1).expand(N, C, H, W).contiguous()
    dx = torch.empty((N, C, H, W), dtype=dy.dtype, device=dy.device, memory_format=torch.channels_last)
    _check(lib().tepd_gap_bwd_nhwc(dy.contiguous().data_ptr(), dx.data_ptr(), N, H * W, C, _stream()), "gap_bwd")
    _count()
    return dx


def bn_native_ok(x: torch.Tensor) -> bool:
    return CONV_NATIVE and x.is_cuda and x.dtype == torch.bfloat16 and x.dim() == 4 and x.shape[1] % 8 == 0


def batchnorm_fwd(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float, relu: bool = False):
    """Training-mode batch norm over (N, H, W) of x [N,C,H,W] in channels_last memory -> (y, mean[C], rstd[C])."""
    N, C, H, W = x.shape
    xn = _nhwc(x)
    y = torch.empty_like(xn)
    ws = torch.zeros(2, C, dtype=torch.float32, device=x.device)
    mean = torch.empty(C, dtype=torch.float32, device=x.device)
    rstd = torch.empty(C, dtype=torch.float32, device=x.device)
    _check(lib().tepd_bn_fwd_nhwc(xn.data_ptr(), gamma.data_ptr(), beta.data_ptr(), y.data_ptr(), mean.data_ptr(), rstd.data_ptr(),
                                  ws.data_ptr(), N * H * W, C, float(eps), int(relu), _stream()), "bn_fwd")
    _count(2)
    return y.permute(0, 3, 1, 2), mean, rstd


def batchnorm_bwd(dy: torch.Tensor, x: torch.Tensor, gamma: torch.Tensor, mean: torch.Tensor, rstd: torch.Tensor):
    """-> (dx [N,C,H,W] channels_last, dgamma[C] fp32, dbeta[C] fp32)."""
    N, C, H, W = x.shape
    xn, dyn = _nhwc(x), _nhwc(dy)
    dx = torch.empty_like(xn)
    ws = torch.zeros(2, C, dtype=torch.float32, device=x.device)     # [sum(dy), sum(dy * xhat)] = [dbeta, dgamma]
    _check(lib().tepd_bn_bwd_nhwc(dyn.data_ptr(), xn.data_ptr(), gamma.data_ptr(), mean.data_ptr(), rstd.data_ptr(), dx.data_ptr(),
                                  ws.data_ptr(), N * H * W, C, _stream()), "bn_bwd")
    _count(2)
    return dx.permute(0, 3, 1, 2), ws[1], ws[0]


def batchnorm_fwd_synced(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float, allsum, num_shards: int,
                         relu: bool = False):
    """Synchronised training-mode BatchNorm, native split phases: local per-channel sums (bn_reduce2), `allsum(ws)` completes them
    over the devices that split the batch (one all-reduce of 2 x C floats), apply with the GLOBAL count.  -> (y, mean, rstd)."""
    N, C, H, W = x.shape
    xn = _nhwc(x)
    rows = N * H * W
    y = torch.empty_like(xn)
    ws = torch.zeros(2, C, dtype=torch.float32, device=x.device)
    mean = torch.empty(C, dtype=torch.float32, device=x.device)
    rstd = torch.empty(C, dtype=torch.float32, device=x.device)
    _check(lib().tepd_bn_reduce_nhwc(xn.data_ptr(), None, None, None, ws.data_ptr(), rows, C, 0, _stream()), "bn_reduce")
    allsum(ws)
    _check(lib().tepd_bn_fwd_apply_nhwc(xn.data_ptr(), ws.data_ptr(), gamma.data_ptr(), beta.data_ptr(), y.data_ptr(), mean.data_ptr(),
                                        rstd.data_ptr(), rows, C, float(eps), int(relu), float(rows * num_shards), _stream()), "bn_fwd_apply")
    _count(2)
    return y.permute(0, 3, 1, 2), mean, rstd


def batchnorm_bwd_synced(dy: torch.Tensor, x: torch.Tensor, gamma: torch.Tensor, mean: torch.Tensor, rstd: torch.Tensor, allsum,
                         num_shards: int):
    """-> (dx, dgamma_local, dbeta_local): dgamma / dbeta stay this shard's partial sums (the plan reduces them with the other
    gradients); dx uses the batch-global sums."""
    N, C, H, W = x.shape
    xn, dyn = _nhwc(x), _nhwc(dy)
    rows = N * H * W
    dx = torch.empty_like(xn)
    ws = torch.zeros(2, C, dtype=torch.float32, device=x.device)
    _check(lib().tepd_bn_reduce_nhwc(dyn.data_ptr(), xn.data_ptr(), mean.data_ptr(), rstd.data_ptr(), ws.data_ptr(), rows, C, 1, _stream()),
           "bn_reduce")
    local = ws.clone()
    allsum(ws)
    _check(lib().tepd_bn_bwd_apply_nhwc(dyn.data_ptr(), xn.data_ptr(), gamma.data_ptr(), mean.data_ptr(), rstd.data_ptr(), ws.data_ptr(),
                                        dx.data_ptr(), rows, C, float(rows * num_shards), _stream()), "bn_bwd_apply")
    _count(2)
    return dx.permute(0, 3, 1, 2), local[1], local[0]


# --------------------------------------------------------------------------------------------- LayerNorm
def layernorm_fwd(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5):
    C = x.shape[-1]
    rows = x.numel() // C
    if not x.is_cuda or x.dtype != torch.bfloat16 or C % 8 or C > 4096 or gamma.dtype != torch.float32:
        xf = x.float()
        mean = xf.mean(-1)
        var = xf.var(-1, unbiased=False)
        rstd = torch.rsqrt(var + eps)
        y = ((xf - mean.unsqueeze(-1)) * rstd.unsqueeze(-1) * gamma.float() + beta.float()).to(x.dtype)
        return y, mean.reshape(rows), rstd.reshape(rows)
    x = x.contiguous()
    y = torch.empty_like(x)
    mean = torch.empty(rows, dtype=torch.float32, device=x.device)
    rstd = torch.empty(rows, dtype=torch.float32, device=x.device)
    _check(lib().tepd_layernorm_fwd(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), y.data_ptr(),
                                    mean.data_ptr(), rstd.data_ptr(), rows, C, eps, _stream()), "layernorm_fwd")
    _count()
    return y, mean, rstd


def layernorm_bwd(dy, x, gamma, mean, rstd, dgamma_acc: torch.Tensor, dbeta_acc: torch.Tensor,
                  dres: Optional[torch.Tensor] = None):
    """Returns dx (+ dres when given: fused residual-stream gradient add); accumulates dgamma/dbeta (fp32)."""
    C = x.shape[-1]
    rows = x.numel() // C
    if not x.is_cuda or x.dtype != torch.bfloat16 or C % 8 or C > 2048 or gamma.dtype != torch.float32:
        xf, dyf = x.float().reshape(rows, C), dy.float().reshape(rows, C)
        xh = (xf - mean.unsqueeze(-1)) * rstd.unsqueeze(-1)
        g = dyf * gamma.float()
        dx = rstd.unsqueeze(-1) * (g - g.mean(-1, keepdim=True) - xh * (g * xh).mean(-1, keepdim=True))
        dgamma_acc.add_((dyf * xh).sum(0))
        dbeta_acc.add_(dyf.sum(0))
        if dres is not None:
            dx = dx + dres.float().reshape(rows, C)
        return dx.to(x.dtype).reshape(x.shape)
    dy = dy.contiguous()
    dx = torch.empty_like(x)
    _check(lib().tepd_layernorm_bwd(dy.data_ptr(), x.data_ptr(), gamma.data_ptr(), mean.data_ptr(), rstd.data_ptr(),
                                    dx.data_ptr(), dgamma_acc.data_ptr(), dbeta_acc.data_ptr(),
                                    None if dres is None else dres.contiguous().data_ptr(), rows, C, _stream()),
           "layernorm_bwd")
    _count()
    return dx


# --------------------------------------------------------------------------------------------- GELU / colsum
def gelu_fwd(x: torch.Tensor) -> torch.Tensor:
    if not x.is_cuda or x.dtype != torch.bfloat16 or x.numel() % 8:
        return torch.nn.functional.gelu(x.float(), approximate="tanh").to(x.dtype)
    x = x.contiguous()
    y = torch.empty_like(x)
    _check(lib().tepd_gelu_fwd(x.data_ptr(), y.data_ptr(), x.numel(), _stream()), "gelu_fwd")
    _count()
    return y


def gelu_bwd(dy: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    if not x.is_cuda or x.dtype != torch.bfloat16 or dy.dtype != torch.bfloat16 or x.numel() % 8:
        xf = x.float().detach().requires_grad_(True)
        with torch.enable_grad():
            y = torch.nn.functional.gelu(xf, approximate="tanh")
        (g,) = torch.autograd.grad(y, xf, dy.float())
        return g.to(x.dtype)
    dy = dy.contiguous()
    dx = torch.empty_like(x)
    _check(lib().tepd_gelu_bwd(dy.data_ptr(), x.data_ptr(), dx.data_ptr(), x.numel(), _stream()), "gelu_bwd")
    _count()
    return dx


def colsum_acc(x: torch.Tensor, out_acc: torch.Tensor) -> None:
    """out_acc[c] += sum_r x[r, c] (bias gradients, fp32 accumulate)."""
    C = x.shape[-1]
    rows = x.numel() // C
    if not x.is_cuda or x.dtype != torch.bfloat16 or C % 8:
        out_acc.add_(x.float().reshape(rows, C).sum(0))
        return
    x = x.contiguous()
    _check(lib().tepd_colsum(x.data_ptr(), out_acc.data_ptr(), rows, C, _stream()), "colsum")
    _count()


# --------------------------------------------------------------------------------------------- embedding
def embedding_fwd(tokens: torch.Tensor, wte: torch.Tensor, wpe: torch.Tensor) -> torch.Tensor:
    B, S = tokens.shape
    C = wte.shape[1]
    if not tokens.is_cuda:
        pos = torch.arange(S, device=tokens.device)
        return (wte[tokens.long()].float() + wpe[pos].float()).to(wte.dtype)
    out = torch.empty(B, S, C, dtype=wte.dtype, device=wte.device)
    tok = tokens.to(torch.int32).contiguous()
    _check(lib().tepd_embedding_fwd(tok.data_ptr(), wte.data_ptr(), wpe.data_ptr(), out.data_ptr(), B * S, S, C,
                                    _stream()), "embedding_fwd")
    _count()
    return out


def embedding_bwd(tokens: torch.Tensor, dout: torch.Tensor, dwte_acc: torch.Tensor, dwpe_acc: torch.Tensor) -> None:
    B, S = tokens.shape
    C = dout.shape[-1]
    if not tokens.is_cuda:
        d = dout.float().reshape(B * S, C)
        dwte_acc.index_add_(0, tokens.reshape(-1).long(), d)
        dwpe_acc[:S].add_(dout.float().reshape(B, S, C).sum(0))
        return
    tok = tokens.to(torch.int32).contiguous()
    dout = dout.contiguous()
    _check(lib().tepd_embedding_bwd(tok.data_ptr(), dout.data_ptr(), dwte_acc.data_ptr(), dwpe_acc.data_ptr(), B * S, S,
                                    C, _stream()), "embedding_bwd")
    _count()


# --------------------------------------------------------------------------------------------- loss
def xent_fwd_bwd(logits: torch.Tensor, labels: torch.Tensor, vocab: int, grad_scale: float):
    """Fused softmax-cross-entropy.  ``logits`` [T, Vp] is overwritten with d(loss)/d(logits)*grad_scale
    (columns >= vocab get zero).  Returns (sum(loss)*grad_scale as 1-elem fp32 tensor, per-row loss)."""
    T, Vp = logits.shape
    if not logits.is_cuda:
        lf = logits.float()[:, :vocab]
        lse = torch.logsumexp(lf, -1)
        rows = lse - lf.gather(1, labels.long().unsqueeze(1)).squeeze(1)
        p = torch.softmax(lf, -1)
        p[torch.arange(T), labels.long()] -= 1.0
        g = torch.zeros(T, Vp)
        g[:, :vocab] = p * grad_scale
        logits.copy_(g.to(logits.dtype))
        return (rows.sum() * grad_scale).reshape(1), rows
    assert logits.is_contiguous() and logits.dtype == torch.bfloat16
    lab = labels.to(torch.int32).contiguous()
    rows = torch.empty(T, dtype=torch.float32, device=logits.device)
    total = torch.zeros(1, dtype=torch.float32, device=logits.device)
    _check(lib().tepd_xent_fwd_bwd(logits.data_ptr(), lab.data_ptr(), rows.data_ptr(), total.data_ptr(), T, vocab, Vp,
                                   grad_scale, _stream()), "xent_fwd_bwd")
    _count()
    return total, rows


# --------------------------------------------------------------------------------------------- optimizer
def adamw_step(p: torch.Tensor, g: torch.Tensor, m: torch.Tensor, v: torch.Tensor, p_bf16: Optional[torch.Tensor],
               n_decay: int, lr: float, beta1: float, beta2: float, eps: float, wd: float, step: int,
               grad_scale: float = 1.0, hyper: Optional[torch.Tensor] = None) -> None:
    """Fused AdamW over flat fp32 buffers (decay applies to the prefix [0, n_decay)).
    ``hyper`` (device fp32 [4] = lr, bc1, bc2, grad_scale) overrides the scalars: CUDA-graph friendly."""
    bc1 = 1.0 - beta1 ** step
    bc2 = 1.0 - beta2 ** step
    n = p.numel()
    if not p.is_cuda:
        if hyper is not None:
            lr, bc1, bc2, grad_scale = (float(x) for x in hyper[:4].tolist())
        gr = g * grad_scale
        m.mul_(beta1).add_(gr, alpha=1 - beta1)
        v.mul_(beta2).addcmul_(gr, gr, value=1 - beta2)
        upd = (m / bc1) / ((v / bc2).sqrt() + eps)
        decay = torch.zeros_like(p)
        decay[:n_decay] = wd
        p.sub_(lr * (upd + decay * p))
        if p_bf16 is not None:
            p_bf16.copy_(p.to(p_bf16.dtype))
        return
    _check(lib().tepd_adamw(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), _p(p_bf16), n, n_decay,
                            lr, beta1, beta2, eps, wd, bc1, bc2, grad_scale, _p(hyper), _stream()), "adamw")
    _count()


def sgd_step(p: torch.Tensor, g: torch.Tensor, p_bf16: Optional[torch.Tensor], lr: float, grad_scale: float = 1.0):
    if not p.is_cuda:
        p.sub_(lr * grad_scale * g)
        if p_bf16 is not None:
            p_bf16.copy_(p.to(p_bf16.dtype))
        return
    _check(lib().tepd_sgd(p.data_ptr(), g.data_ptr(), _p(p_bf16), p.numel(), lr, grad_scale, _stream()), "sgd")
    _count()


def axpy_f32(acc: torch.Tensor, g: torch.Tensor, a: float = 1.0) -> None:
    if not acc.is_cuda:
        acc.add_(g, alpha=a)
        return
    _check(lib().tepd_axpy_f32(acc.data_ptr(), g.data_ptr(), acc.numel(), a, _stream()), "axpy_f32")
    _count()


def cast_f32_bf16(src: torch.Tensor, dst: torch.Tensor) -> None:
    if not src.is_cuda:
        dst.copy_(src.to(dst.dtype))
        return
    _check(lib().tepd_cast_f32_bf16(src.data_ptr(), dst.data_ptr(), src.numel(), _stream()), "cast_f32_bf16")
    _count()


# --------------------------------------------------------------------------------------------- attention
from .attention import attention_fwd, attention_bwd  # noqa: E402,F401
