"""torch-tensor front end of the C-ABI (include/vl2.h).  Every function enqueues libvl2 kernels on the current CUDA
stream and returns the output tensor; nothing here computes with torch ops (torch only owns memory and streams)."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

from . import _lib
from ._lib import (ACT_GELU_ERF, ACT_GELU_TANH, ACT_NONE, ACT_QUICK_GELU, ACT_SIGMOID, ACT_SILU, ACT_SWIGLU, AttnArgs, GemmArgs,
                   check)

__all__ = [
    "gemm", "gemm_skinny", "attention", "attention_decode", "decode_rope_append", "attention_decode_dyn", "gemv", "quantize_fp8_rows", "decode_workspace", "l2_prefetch", "layernorm", "rmsnorm", "row_sumsq", "row_stats", "patch_im2col", "patch_embed", "clip_embed_finish",
    "dwconv3x3_ln_silu", "se_scale", "conv3d_im2col", "conv3d_k2s2", "rope_inplace", "embed_splice", "launch_count",
    "ACT_NONE", "ACT_QUICK_GELU", "ACT_SILU", "ACT_GELU_ERF", "ACT_GELU_TANH", "ACT_SWIGLU", "ACT_SIGMOID",
]


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _need_cuda(*ts: Optional[torch.Tensor]) -> None:
    """Every operand must live on the CURRENT CUDA device: the kernels are enqueued on that device's current stream
    (`_stream`), so a tensor of another GPU would be dereferenced from the wrong device.  Callers that drive several GPUs
    from one process wrap the call in `torch.cuda.device(i)` (the engine classes do: model/_device_guard)."""
    cur = None
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise _lib.Vl2Error("videollama2_b200 kernels need CUDA tensors; there is no CPU fallback")
        if cur is None:
            cur = torch.cuda.current_device()
        if t.device.index != cur:
            raise _lib.Vl2Error(f"tensor on cuda:{t.device.index} but the current device is cuda:{cur}: run the call under "
                                f"`torch.cuda.device({t.device.index})` (kernels launch on the current device's stream)")


_STORAGE = (torch.bfloat16, torch.float16)


def _bf16(*ts: Optional[torch.Tensor]) -> None:
    """All given tensors hold the library's 16-bit storage type: bfloat16 (libvl2.so) or float16 (libvl2_f16.so), and the
    same one - the two builds are separate libraries and a call runs entirely in one of them."""
    dt = None
    for t in ts:
        if t is None:
            continue
        if t.dtype not in _STORAGE:
            raise TypeError(f"expected a bfloat16 / float16 tensor, got {t.dtype}")
        if dt is None:
            dt = t.dtype
        elif t.dtype != dt:
            raise TypeError(f"mixed storage types in one call: {dt} and {t.dtype}")


def _L(t: torch.Tensor):
    """The build of the library that matches tensor t's storage type."""
    return _lib.load(t.dtype)


def launch_count() -> int:
    """Kernel launches issued by the library (both storage-type builds) in this process."""
    _lib.load()
    return sum(int(l.vl2_launch_count()) for l in _lib._libs.values())


def gemm(a: torch.Tensor, w: torch.Tensor, *, bias: Optional[torch.Tensor] = None, act: int = ACT_NONE,
         residual: Optional[torch.Tensor] = None, row_scale: Optional[torch.Tensor] = None,
         out: Optional[torch.Tensor] = None, out_dtype: Optional[torch.dtype] = None, bn: int = 0,
         bcast_ptrs: Optional[list] = None, mc_ptr: int = 0, rms_in: Optional[torch.Tensor] = None,
         rms_eps: float = 0.0, sumsq_out: Optional[torch.Tensor] = None, trace: bool = False,
         splitk=True, ln_in=None, ln_colsum: Optional[torch.Tensor] = None,
         rowsum_out: Optional[torch.Tensor] = None, rope=None, general_epilogue: bool = False) -> torch.Tensor:
    """out[M,Nout] = epi(a[M,K] @ w[N,K]^T); a/w may be row-strided views (last dim contiguous).
    `bn` forces the tile width (tests); 0 = library heuristic.
    `bcast_ptrs`: device pointers of peer buffers (same layout as `out`) that receive every output vector too
    (epilogue-fused all-gather over NVLink); `mc_ptr`: NVSwitch multicast address used instead when non-zero.
    `rms_in` (fp32 [M, parts] partial row sums of squares of `a`) scales row m by rsqrt(sum(rms_in[m])/K + rms_eps):
    RMSNorm folded into the GEMM (gamma must already be folded into w); `sumsq_out` (fp32 [M, N/32]) receives the
    per-32-column sums of squares of the bf16 outputs (no atomics: bit-reproducible).
    `ln_in` = (row sums, row sums of squares) of `a`, both fp32 [M, parts], with `ln_colsum` (fp32 [N] = sum_k w[n,k]):
    LayerNorm folded into the GEMM (gamma folded into w, beta into bias; eps = `rms_eps`):
    rstd * (a w^T - mu * colsum) + bias.  `rowsum_out` (fp32 [M, N/32], together with `sumsq_out`): per-32-column sums of
    the bf16 outputs, i.e. the statistics the NEXT folded LayerNorm needs.
    `general_epilogue` (tests): run the kernel's general epilogue where the lean one (TMA stores) would be picked."""
    _need_cuda(a, w, bias, residual, row_scale, out)
    _bf16(a, w, residual)
    assert a.dim() == 2 and w.dim() == 2 and a.stride(1) == 1 and w.stride(1) == 1, "gemm: 2-D, unit inner stride"
    M, K = a.shape
    N, Kw = w.shape
    if K != Kw:
        raise ValueError(f"gemm: K mismatch {K} vs {Kw}")
    n_out = N // 2 if act == ACT_SWIGLU else N
    if out is None:
        out = torch.empty((M, n_out), device=a.device, dtype=out_dtype or a.dtype)
    assert out.shape == (M, n_out) and out.stride(1) == 1
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.numel() == N and bias.is_contiguous()
    if residual is not None:
        assert residual.shape == (M, n_out) and residual.stride(1) == 1
    if row_scale is not None:
        assert row_scale.dtype == torch.float32 and row_scale.numel() == M and row_scale.is_contiguous()
    args = GemmArgs(A=a.data_ptr(), W=w.data_ptr(), C=out.data_ptr(), bias=_ptr(bias), residual=_ptr(residual),
                    row_scale=_ptr(row_scale), lda=a.stride(0), ldw=w.stride(0), ldc=out.stride(0),
                    ldr=residual.stride(0) if residual is not None else 0, M=M, N=N, K=K, act=act,
                    out_f32=1 if out.dtype == torch.float32 else 0, reserved=bn)
    if out.dtype not in (torch.float32, a.dtype):
        raise TypeError("gemm: out must have the operands' storage type or be fp32")
    if rms_in is not None:
        assert rms_in.is_cuda and rms_in.dtype == torch.float32 and rms_in.is_contiguous() and rms_in.shape[0] == M
        args.rms_sumsq_in = rms_in.data_ptr()
        args.rms_nparts = rms_in.numel() // M
        args.rms_inv_dim = 1.0 / K
        args.rms_eps = float(rms_eps)
    if rope is not None:
        # (table uint32 [positions, D/2] packed bf16 cos|sin, first position, head width D, number of leading q/k columns):
        # RoPE applied in the epilogue to adjacent column pairs (weights permuted accordingly, see rope_interleave_rows)
        tab, pos0, hd, cols = rope
        _need_cuda(tab)
        assert tab.dtype == torch.int32 and tab.is_contiguous() and tab.shape[1] == hd // 2 and tab.shape[0] >= pos0 + M
        args.rope_tab = tab.data_ptr()
        args.rope_cols, args.rope_D, args.rope_pos0 = int(cols), int(hd), int(pos0)
    if ln_in is not None:
        if rms_in is not None or ln_colsum is None:
            raise ValueError("gemm: ln_in excludes rms_in and needs ln_colsum")
        ln_sum, ln_sq = ln_in
        for t in (ln_sum, ln_sq):
            assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.shape[0] == M
        assert ln_sum.shape == ln_sq.shape and ln_colsum.dtype == torch.float32 and ln_colsum.numel() == N and ln_colsum.is_contiguous()
        _need_cuda(ln_sum, ln_sq, ln_colsum)
        args.ln_sum_in = ln_sum.data_ptr()
        args.rms_sumsq_in = ln_sq.data_ptr()
        args.ln_colsum = ln_colsum.data_ptr()
        args.rms_nparts = ln_sq.numel() // M
        args.rms_inv_dim = 1.0 / K
        args.rms_eps = float(rms_eps)
    if rowsum_out is not None:
        if sumsq_out is None:
            raise ValueError("gemm: rowsum_out is written together with sumsq_out")
        assert rowsum_out.is_cuda and rowsum_out.dtype == torch.float32 and rowsum_out.is_contiguous()
        assert tuple(rowsum_out.shape) == (M, N // 32)
        args.rowsum_out = rowsum_out.data_ptr()
    if sumsq_out is not None:
        if out.dtype == torch.float32 or act == ACT_SWIGLU or N % 32:
            raise NotImplementedError("gemm: sumsq_out supports 16-bit, non-SwiGLU outputs with N % 32 == 0")
        assert sumsq_out.is_cuda and sumsq_out.dtype == torch.float32 and sumsq_out.is_contiguous()
        assert tuple(sumsq_out.shape) == (M, N // 32)
        args.sumsq_out = sumsq_out.data_ptr()
    if bcast_ptrs or mc_ptr:
        if out.dtype == torch.float32 or act == ACT_SWIGLU:
            raise NotImplementedError("gemm: broadcast epilogue supports 16-bit, non-SwiGLU outputs")
        ptrs = list(bcast_ptrs or [])
        if len(ptrs) > 8:
            raise ValueError("gemm: at most 8 broadcast targets")
        for i, ptr in enumerate(ptrs):
            args.bcast_out[i] = ptr
        args.n_bcast = len(ptrs)
        args.mc_out = mc_ptr or None
    if trace:
        args.reserved2 = 777
    if general_epilogue:
        args.reserved4 = 1                          # test hook: the general epilogue instead of the lean (TMA-store) one
    forced = splitk is not True and splitk and int(splitk) > 1
    if forced or (splitk and _SPLITK_ENV):          # the workspace exists only when the split-K tail can actually run
        if forced:
            args.reserved3 = int(splitk)            # test hook: force the number of K-slices
        ws = _splitk_workspace(a.device)
        args.splitk_ws = ws.data_ptr()
        args.splitk_ws_bytes = ws.numel()
    check(_L(a).vl2_gemm_bf16(C.byref(args), _stream()), "vl2_gemm_bf16")
    return out


_SPLITK_WS_BYTES = 48 << 20
_SPLITK_ENV = os.environ.get("VL2_GEMM_SPLITK", "0") == "1"   # same switch as the library's splitk_enabled()
_splitk_ws = {}


def _splitk_workspace(device) -> torch.Tensor:
    """Per-(device, stream) split-K scratch of vl2_gemm_bf16 (zero-filled once: its counters re-arm themselves)."""
    key = (torch.device(device).index, _stream())
    ws = _splitk_ws.get(key)
    if ws is None:
        ws = torch.zeros((_SPLITK_WS_BYTES,), device=device, dtype=torch.uint8)
        _splitk_ws[key] = ws
    return ws


def gemm_trace() -> list:
    """Tile-boundary cycle trace of the last gemm(..., trace=True) launch (vl2_debug_gemm_trace)."""
    buf = (C.c_longlong * 128)()
    check(_lib.load().vl2_debug_gemm_trace(buf), "vl2_debug_gemm_trace")
    return list(buf)


def gemm_skinny(a: torch.Tensor, w: torch.Tensor, *, bias: Optional[torch.Tensor] = None, act: int = ACT_NONE,
                residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
                out_dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """out[M,Nout] = act(a[M,K] @ w[N,K]^T + bias) (+ residual), M <= 32; weight-streaming (decode / SE / lm_head)."""
    _need_cuda(a, w, bias, residual, out)
    _bf16(w, residual)
    assert a.is_contiguous() and w.is_contiguous() and a.dim() == 2 and w.dim() == 2
    M, K = a.shape
    N = w.shape[0]
    assert w.shape[1] == K
    assert a.dtype in (torch.float32, w.dtype)
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.numel() == N
    n_out = N // 2 if act == ACT_SWIGLU else N
    if out is None:
        out = torch.empty((M, n_out), device=a.device, dtype=out_dtype)
    assert out.is_contiguous() and out.numel() == M * n_out and out.dtype in (torch.float32, w.dtype)
    if residual is not None:
        assert residual.is_contiguous() and residual.numel() == M * n_out
    check(_L(w).vl2_gemm_skinny(a.data_ptr(), 1 if a.dtype == torch.float32 else 0, w.data_ptr(), _ptr(bias),
                                      _ptr(residual), out.data_ptr(), 1 if out.dtype == torch.float32 else 0, M, N, K,
                                      act, _stream()), "vl2_gemm_skinny")
    return out


class pdl:
    """Context manager: programmatic dependent launch for the vl2 launches inside (vl2_set_pdl)."""

    def __init__(self, on: bool = True):
        self.on = on

    def __enter__(self):
        _lib.load()
        for lib in _lib._libs.values():
            check(lib.vl2_set_pdl(1 if self.on else 0), "vl2_set_pdl")
        return self

    def __exit__(self, *exc):
        for lib in _lib._libs.values():
            check(lib.vl2_set_pdl(-1), "vl2_set_pdl")
        return False


def l2_prefetch(t: torch.Tensor, nbytes: Optional[int] = None) -> None:
    """Hint the first `nbytes` of a contiguous device tensor of any dtype (e.g. fp8 decode weights) into L2
    (vl2_l2_prefetch) on the current stream."""
    _need_cuda(t)
    total = t.numel() * t.element_size()
    n = total if nbytes is None else min(int(nbytes), total)
    # a byte-level kernel, the same in both builds: a 16-bit tensor uses its own build, any other dtype (fp8 weights) a
    # build this process already loaded, so that an fp16 model does not load the bf16 library only for this call
    if t.dtype in _STORAGE:
        lib = _L(t)
    else:
        lib = next(iter(_lib._libs.values())) if _lib._libs else _lib.load()
    check(lib.vl2_l2_prefetch(t.data_ptr(), n, _stream()), "vl2_l2_prefetch")


_decode_ws = {}


def decode_workspace(device, Hq: int, Hkv: int, D: int) -> torch.Tensor:
    """Per-(device, stream) scratch for the split-KV decode attention (vl2_attention_decode_workspace bytes)."""
    key = (torch.device(device).index, _stream(), Hq, Hkv, D)
    ws = _decode_ws.get(key)
    if ws is None:
        nbytes = int(_lib.load().vl2_attention_decode_workspace(Hq, Hkv, D))
        ws = torch.empty((nbytes // 4,), device=device, dtype=torch.float32)
        _decode_ws[key] = ws
    return ws


FP8_MAX = 448.0   # largest finite float8_e4m3fn value


def quantize_fp8_rows(w: torch.Tensor):
    """w [N,K] (any float dtype) -> (w8 float8_e4m3fn [N,K], scale fp32 [N]) with w ~= w8 * scale[:, None]: one scale per
    output row, amax_row / 448 (1 for an all-zero row), round-to-nearest-even after clamping to +-448 so that no NaN
    code (0x7F / 0xFF) appears.  Load-time weight preparation for the fp8 decode GEMV (vl2_gemv_fp8), in plain torch."""
    assert w.dim() == 2
    wf = w.float()
    amax = wf.abs().amax(dim=1)
    scale = torch.where(amax > 0, amax / FP8_MAX, torch.ones_like(amax))
    w8 = (wf / scale[:, None]).clamp_(-FP8_MAX, FP8_MAX).to(torch.float8_e4m3fn)
    return w8.contiguous(), scale.contiguous()


def gemv(x: torch.Tensor, w: torch.Tensor, *, bias: Optional[torch.Tensor] = None, act: int = ACT_NONE,
         residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None, rms_eps: float = 0.0,
         out_dtype: Optional[torch.dtype] = None, w_scale: Optional[torch.Tensor] = None) -> torch.Tensor:
    """y[1,Nout] = act(s * w[N,K] x + bias) (+ residual); rms_eps > 0 fuses the RMSNorm in front (gain folded into w).
    A float8_e4m3fn `w` (from quantize_fp8_rows) needs its per-row fp32 `w_scale` [N] and runs vl2_gemv_fp8."""
    fp8 = w.dtype == torch.float8_e4m3fn
    if fp8 != (w_scale is not None):
        raise ValueError("gemv: a float8_e4m3fn weight needs w_scale, and only such a weight takes one")
    _need_cuda(x, w, bias, residual, out, w_scale)
    _bf16(x, None if fp8 else w, residual)
    assert x.is_contiguous() and w.is_contiguous() and w.dim() == 2 and x.numel() == w.shape[1]
    N, K = w.shape
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.numel() == N
    if fp8:
        assert w_scale.dtype == torch.float32 and w_scale.is_contiguous() and w_scale.numel() == N
    n_out = N // 2 if act == ACT_SWIGLU else N
    if out is None:
        out = torch.empty((1, n_out), device=x.device, dtype=out_dtype or x.dtype)
    assert out.is_contiguous() and out.numel() == n_out and out.dtype in (torch.float32, x.dtype)
    if residual is not None:
        assert residual.is_contiguous() and residual.numel() == n_out
    out_f32 = 1 if out.dtype == torch.float32 else 0
    if fp8:
        check(_L(x).vl2_gemv_fp8(x.data_ptr(), w.data_ptr(), w_scale.data_ptr(), _ptr(bias), _ptr(residual),
                                 out.data_ptr(), out_f32, N, K, act, float(rms_eps), _stream()), "vl2_gemv_fp8")
    else:
        check(_L(w).vl2_gemv_bf16(x.data_ptr(), w.data_ptr(), _ptr(bias), _ptr(residual), out.data_ptr(),
                                  out_f32, N, K, act, float(rms_eps), _stream()), "vl2_gemv_bf16")
    return out


def attention_decode(q: torch.Tensor, k_cache: torch.Tensor, v_cache: torch.Tensor, *, n_pos: int, Hq: int, Hkv: int,
                     D: int, scale: float, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """q [Hq*D]; k_cache / v_cache: row-strided views [>=n_pos, Hkv*D] of the per-layer cache."""
    _need_cuda(q, k_cache, v_cache)
    _bf16(q, k_cache, v_cache)
    assert q.is_contiguous() and q.numel() == Hq * D and k_cache.stride(1) == 1 and v_cache.stride(1) == 1
    assert k_cache.stride(0) == v_cache.stride(0) and k_cache.shape[0] >= n_pos
    if out is None:
        out = torch.empty((1, Hq * D), device=q.device, dtype=q.dtype)
    ws = decode_workspace(q.device, Hq, Hkv, D)
    check(_L(k_cache).vl2_attention_decode(q.data_ptr(), k_cache.data_ptr(), v_cache.data_ptr(), out.data_ptr(),
                                           k_cache.stride(0), n_pos, Hq, Hkv, D, float(scale), ws.data_ptr(), _stream()),
          "vl2_attention_decode")
    return out


def attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, *, B: int, S: int, Hq: int, Hkv: int, D: int,
              causal: bool, scale: float, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """q/k/v: 2-D row-strided views [B*S, H*D] (e.g. column slices of a fused QKV buffer)."""
    _need_cuda(q, k, v, out)
    _bf16(q, k, v)
    for t, h in ((q, Hq), (k, Hkv), (v, Hkv)):
        assert t.dim() == 2 and t.shape == (B * S, h * D) and t.stride(1) == 1
    if out is None:
        out = torch.empty((B * S, Hq * D), device=q.device, dtype=q.dtype)
    args = AttnArgs(q=q.data_ptr(), k=k.data_ptr(), v=v.data_ptr(), out=out.data_ptr(), ldq=q.stride(0),
                    ldk=k.stride(0), ldv=v.stride(0), ldo=out.stride(0), B=B, S=S, Hq=Hq, Hkv=Hkv, D=D,
                    causal=1 if causal else 0, scale=float(scale), reserved=0)
    check(_L(q).vl2_attention(C.byref(args), _stream()), "vl2_attention")
    return out


def decode_rope_append(qkv_row: torch.Tensor, cache: torch.Tensor, pos_dev: torch.Tensor, Hq: int, Hkv: int, D: int,
                       inv_freq: torch.Tensor, interleaved: bool = False) -> None:
    """Graph-replayable: rotate q/k of the fused row at position *pos_dev and append the row to cache[*pos_dev]."""
    _need_cuda(qkv_row, cache, pos_dev, inv_freq)
    _bf16(qkv_row, cache)
    assert qkv_row.is_contiguous() and qkv_row.numel() == (Hq + 2 * Hkv) * D and cache.stride(1) == 1
    assert pos_dev.dtype == torch.int32 and pos_dev.numel() == 1
    check(_L(qkv_row).vl2_decode_rope_append(qkv_row.data_ptr(), cache.data_ptr(), cache.stride(0), pos_dev.data_ptr(),
                                             Hq, Hkv, D, inv_freq.data_ptr(), 1 if interleaved else 0, _stream()),
          "vl2_decode_rope_append")


def attention_decode_dyn(q: torch.Tensor, k_cache: torch.Tensor, v_cache: torch.Tensor, pos_dev: torch.Tensor, *,
                         Hq: int, Hkv: int, D: int, scale: float, out: torch.Tensor,
                         workspace: Optional[torch.Tensor] = None) -> torch.Tensor:
    _need_cuda(q, k_cache, v_cache, pos_dev, out)
    _bf16(q, k_cache, v_cache, out)
    assert k_cache.stride(0) == v_cache.stride(0) and pos_dev.dtype == torch.int32
    ws = workspace if workspace is not None else decode_workspace(q.device, Hq, Hkv, D)
    check(_L(q).vl2_attention_decode_dyn(q.data_ptr(), k_cache.data_ptr(), v_cache.data_ptr(), out.data_ptr(),
                                               k_cache.stride(0), pos_dev.data_ptr(), Hq, Hkv, D, float(scale),
                                               ws.data_ptr(), _stream()), "vl2_attention_decode_dyn")
    return out


def layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float, *, act: int = ACT_NONE,
              residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _need_cuda(x, gamma, beta, residual, out)
    _bf16(x, gamma, beta, residual)
    assert x.is_contiguous()
    Cc = x.shape[-1]
    rows = x.numel() // Cc
    if out is None:
        out = torch.empty_like(x)
    if residual is not None:
        assert residual.is_contiguous() and residual.shape == x.shape
    check(_L(x).vl2_layernorm(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), _ptr(residual), out.data_ptr(),
                                    rows, Cc, float(eps), act, _stream()), "vl2_layernorm")
    return out


def rmsnorm(x: torch.Tensor, gamma: torch.Tensor, eps: float, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _need_cuda(x, gamma, out)
    _bf16(x, gamma)
    assert x.is_contiguous()
    Cc = x.shape[-1]
    if out is None:
        out = torch.empty_like(x)
    check(_L(x).vl2_rmsnorm(x.data_ptr(), gamma.data_ptr(), out.data_ptr(), x.numel() // Cc, Cc, float(eps),
                                  _stream()), "vl2_rmsnorm")
    return out


def row_stats(x: torch.Tensor):
    """(sum, sum of squares) of every row of x [rows, C], each fp32 [rows, 1]: the statistics a folded LayerNorm reads
    when its input does not come out of a GEMM epilogue."""
    _need_cuda(x)
    _bf16(x)
    assert x.is_contiguous() and x.dim() == 2
    s = torch.empty((x.shape[0], 1), device=x.device, dtype=torch.float32)
    q = torch.empty((x.shape[0], 1), device=x.device, dtype=torch.float32)
    check(_L(x).vl2_row_stats(x.data_ptr(), s.data_ptr(), q.data_ptr(), x.shape[0], x.shape[1], _stream()), "vl2_row_stats")
    return s, q


def row_sumsq(x: torch.Tensor) -> torch.Tensor:
    _need_cuda(x)
    _bf16(x)
    assert x.is_contiguous() and x.dim() == 2
    out = torch.empty((x.shape[0], 1), device=x.device, dtype=torch.float32)
    check(_L(x).vl2_row_sumsq(x.data_ptr(), out.data_ptr(), x.shape[0], x.shape[1], _stream()), "vl2_row_sumsq")
    return out


def patch_im2col(pixels: torch.Tensor, P: int, Kpad: int) -> torch.Tensor:
    _need_cuda(pixels)
    _bf16(pixels)
    assert pixels.is_contiguous() and pixels.dim() == 4 and pixels.shape[1] == 3
    F, _, H, W = pixels.shape
    out = torch.empty((F * (H // P) * (W // P), Kpad), device=pixels.device, dtype=pixels.dtype)
    check(_L(pixels).vl2_patch_im2col(pixels.data_ptr(), out.data_ptr(), F, H, W, P, Kpad, _stream()),
          "vl2_patch_im2col")
    return out


def patch_embed(pixels: torch.Tensor, weight: torch.Tensor, pos: torch.Tensor, P: int, *, cls: Optional[torch.Tensor] = None,
                gamma: Optional[torch.Tensor] = None, beta: Optional[torch.Tensor] = None, bias: Optional[torch.Tensor] = None,
                eps: float = 1e-5) -> torch.Tensor:
    """ViT embeddings in one implicit-GEMM launch (vl2_patch_embed).  CLIP form (cls / gamma / beta given): class token +
    patch conv + positions + pre-LayerNorm -> [F*(np+1), C]; SigLIP form (bias given): conv + bias + positions -> [F*np, C].
    weight: [C, Kpad] (conv kernel flattened, zero-padded to a multiple of 64)."""
    _need_cuda(pixels, weight, pos, cls, gamma, beta, bias)
    _bf16(pixels, weight, pos, cls, gamma, beta)
    assert pixels.is_contiguous() and pixels.dim() == 4 and pixels.shape[1] == 3 and weight.is_contiguous() and pos.is_contiguous()
    F, _, H, W = pixels.shape
    Cc, Kpad = weight.shape
    npatch = (H // P) * (W // P)
    clip = gamma is not None
    assert pos.shape == (npatch + (1 if clip else 0), Cc)
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.numel() == Cc
    out = torch.empty((F * (npatch + (1 if clip else 0)), Cc), device=pixels.device, dtype=pixels.dtype)
    a = _lib.PatchEmbedArgs(pixels=pixels.data_ptr(), weight=weight.data_ptr(), pos=pos.data_ptr(), cls=_ptr(cls),
                            gamma=_ptr(gamma), beta=_ptr(beta), bias=_ptr(bias), out=out.data_ptr(), scratch=None,
                            F=F, H=H, W=W, P=P, C=Cc, Kpad=Kpad, eps=float(eps))
    check(_L(pixels).vl2_patch_embed(C.byref(a), _stream()), "vl2_patch_embed")
    return out


def clip_embed_finish(patch: torch.Tensor, cls: torch.Tensor, pos: torch.Tensor, gamma: torch.Tensor,
                      beta: torch.Tensor, F: int, eps: float) -> torch.Tensor:
    _need_cuda(patch, cls, pos, gamma, beta)
    _bf16(patch, cls, pos, gamma, beta)
    assert patch.is_contiguous() and pos.is_contiguous()
    Cc = patch.shape[-1]
    np_ = patch.shape[0] // F
    assert pos.shape == (np_ + 1, Cc)
    out = torch.empty((F * (np_ + 1), Cc), device=patch.device, dtype=patch.dtype)
    check(_L(patch).vl2_clip_embed_finish(patch.data_ptr(), cls.data_ptr(), pos.data_ptr(), gamma.data_ptr(),
                                            beta.data_ptr(), out.data_ptr(), F, np_, Cc, float(eps), _stream()),
          "vl2_clip_embed_finish")
    return out


def dwconv3x3_ln_silu(x: torch.Tensor, w9c: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float,
                      with_pool: bool = True):
    """x: [F,H,W,C] channels-last bf16.  Returns (y, pooled[F,C] fp32 or None)."""
    _need_cuda(x, w9c, gamma, beta)
    _bf16(x, w9c, gamma, beta)
    assert x.is_contiguous() and x.dim() == 4 and w9c.is_contiguous() and w9c.shape == (9, x.shape[-1])
    F, H, W, Cc = x.shape
    y = torch.empty_like(x)
    pool = torch.empty((F * Cc + F * H * Cc,), device=x.device, dtype=torch.float32) if with_pool else None
    check(_L(x).vl2_dwconv3x3_ln_silu(x.data_ptr(), w9c.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                                            y.data_ptr(), _ptr(pool), F, H, W, Cc, float(eps), _stream()),
          "vl2_dwconv3x3_ln_silu")
    return y, (pool[: F * Cc].view(F, Cc) if with_pool else None)


def se_scale(y: torch.Tensor, s: torch.Tensor) -> torch.Tensor:
    """In place: y[f, :, :, c] *= s[f, c]."""
    _need_cuda(y, s)
    _bf16(y)
    assert y.is_contiguous() and s.dtype == torch.float32 and s.is_contiguous()
    F, Cc = s.shape
    HW = y.numel() // (F * Cc)
    check(_L(y).vl2_se_scale(y.data_ptr(), s.data_ptr(), F, HW, Cc, _stream()), "vl2_se_scale")
    return y


def conv3d_k2s2(x: torch.Tensor, w: torch.Tensor, *, bias: Optional[torch.Tensor] = None, act: int = ACT_NONE, pad: int = 1,
                out: Optional[torch.Tensor] = None, bn: int = 0) -> torch.Tensor:
    """nn.Conv3d(C, N, kernel_size=2, stride=2, padding=pad) (+bias, +activation) on channels-last x [T,H,W,C] as an
    IMPLICIT GEMM: out[(to,ho,wo), N] = act(sum_tap x[2to-pad+dt, 2ho-pad+dh, 2wo-pad+dw, :] w[:, tap*C:(tap+1)*C]^T + bias).
    The GEMM's TMA producer gathers every k-block of every output line straight from x (4-D tensor map, out-of-bounds =
    zero padding); no im2col matrix is materialised.  w: [N, 8*C], K index = tap*C + cin, tap = dt*4 + dh*2 + dw."""
    _need_cuda(x, w, bias, out)
    _bf16(x, w)
    assert x.is_contiguous() and x.dim() == 4 and w.dim() == 2 and w.stride(1) == 1
    T, H, W, Cc = x.shape
    N, K = w.shape
    if K != 8 * Cc:
        raise ValueError(f"conv3d_k2s2: weight K {K} != 8*C {8 * Cc}")
    To, Ho, Wo = (T + 2 * pad - 2) // 2 + 1, (H + 2 * pad - 2) // 2 + 1, (W + 2 * pad - 2) // 2 + 1
    M = To * Ho * Wo
    if out is None:
        out = torch.empty((M, N), device=x.device, dtype=x.dtype)
    assert out.shape == (M, N) and out.stride(1) == 1 and out.dtype == x.dtype
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.numel() == N and bias.is_contiguous()
    args = GemmArgs(A=x.data_ptr(), W=w.data_ptr(), C=out.data_ptr(), bias=_ptr(bias), lda=K, ldw=w.stride(0),
                    ldc=out.stride(0), ldr=0, M=M, N=N, K=K, act=act, out_f32=0, reserved=bn, conv_C=Cc, conv_T=T, conv_H=H,
                    conv_W=W, conv_pad=pad)
    check(_L(x).vl2_gemm_bf16(C.byref(args), _stream()), "vl2_gemm_bf16(conv3d)")
    return out


def conv3d_im2col(x: torch.Tensor, pad: int) -> torch.Tensor:
    """x: [T,H,W,C] -> A [(To*Ho*Wo), 8*C] for the k=s=2 Conv3d with padding `pad`."""
    _need_cuda(x)
    _bf16(x)
    assert x.is_contiguous() and x.dim() == 4
    T, H, W, Cc = x.shape
    To, Ho, Wo = (T + 2 * pad - 2) // 2 + 1, (H + 2 * pad - 2) // 2 + 1, (W + 2 * pad - 2) // 2 + 1
    out = torch.empty((To * Ho * Wo, 8 * Cc), device=x.device, dtype=x.dtype)
    check(_L(x).vl2_conv3d_im2col(x.data_ptr(), out.data_ptr(), T, H, W, Cc, pad, To, Ho, Wo, _stream()),
          "vl2_conv3d_im2col")
    return out


def rope_inplace(qkv: torch.Tensor, S: int, Hq: int, Hkv: int, D: int, q_off: int, k_off: int, pos0: int,
                 inv_freq: torch.Tensor, interleaved: bool = False) -> torch.Tensor:
    _need_cuda(qkv, inv_freq)
    _bf16(qkv)
    assert qkv.dim() == 2 and qkv.stride(1) == 1 and inv_freq.dtype == torch.float32 and inv_freq.numel() == D // 2
    check(_L(qkv).vl2_rope_inplace(qkv.data_ptr(), qkv.stride(0), S, Hq, Hkv, D, q_off, k_off, pos0,
                                       inv_freq.data_ptr(), 1 if interleaved else 0, _stream()), "vl2_rope_inplace")
    return qkv


def rope_interleave_rows(n_heads: int, D: int) -> torch.Tensor:
    """Row permutation of a q / k projection weight [n_heads*D, K] that makes the RoPE partners (i, i + D/2) of every head
    adjacent output columns (2i, 2i+1): new_row[h*D + 2i] = old_row[h*D + i], new_row[h*D + 2i + 1] = old_row[h*D + i + D/2]."""
    i = torch.arange(D // 2)
    per_head = torch.stack([i, i + D // 2], 1).reshape(-1)                       # [D]
    return (torch.arange(n_heads)[:, None] * D + per_head[None, :]).reshape(-1)


def rope_table(n_pos: int, D: int, theta: float, device, dtype: torch.dtype = torch.bfloat16) -> torch.Tensor:
    """[n_pos, D/2] int32: cos (low half) | sin (high half) of angle pos * theta^(-2i/D) as 16-bit values of the storage
    type, computed in fp32 and rounded as HF does before applying them (HF:mistral/modeling_mistral.py:311-324).  Built once
    per engine."""
    inv = 1.0 / (theta ** (torch.arange(0, D, 2, dtype=torch.int64).float() / D))
    ang = torch.outer(torch.arange(n_pos, dtype=torch.float32), inv)
    c = ang.cos().to(dtype).view(torch.int16).to(torch.int32) & 0xFFFF
    sn = ang.sin().to(dtype).view(torch.int16).to(torch.int32) & 0xFFFF
    return (c | (sn << 16)).to(torch.int32).contiguous().to(device)


def embed_splice(ids: torch.Tensor, dst_row: torch.Tensor, table: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    _need_cuda(ids, dst_row, table, out)
    _bf16(table, out)
    assert ids.dtype == torch.int64 and dst_row.dtype == torch.int32 and ids.numel() == dst_row.numel()
    assert table.is_contiguous() and out.is_contiguous() and table.shape[1] == out.shape[1]
    check(_L(table).vl2_embed_splice(ids.data_ptr(), dst_row.data_ptr(), ids.numel(), table.data_ptr(),
                                       table.shape[0], out.data_ptr(), out.shape[1], _stream()), "vl2_embed_splice")
    return out
