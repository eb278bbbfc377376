"""ctypes binding of ``libtensorlink_b200.so`` (the C ABI in ``include/tensorlink_b200.h``).

There is no CPU fallback and no eager-PyTorch twin: if the library is missing, or no sm_100 device is
visible, every compute entry point raises.  PyTorch is used only to own device memory and streams.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_size_t, c_void_p
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libtensorlink_b200.so")

EPI_BIAS, EPI_RESIDUAL, EPI_SWIGLU, EPI_OUT_F32, EPI_ACCUM, A_MN_MAJOR, B_MN_MAJOR = 1, 2, 4, 8, 16, 32, 64


class NativeError(RuntimeError):
    pass


_SIGS = {
    "tl_abi_version": (c_int, []),
    "tl_last_error": (c_char_p, []),
    "tl_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "tl_rmsnorm_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_void_p]),
    "tl_embed_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "tl_gemm_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                             c_void_p, c_void_p, c_int, c_void_p]),
    "tl_gemm_splitk_ws": (c_size_t, [c_int, c_int]),
    "tl_gemm_bf16_ws": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "tl_gemm_bf16_ws_norm": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                     c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_void_p, c_float, c_void_p, c_void_p]),
    "tl_gemv_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                             c_float, c_int, c_void_p]),
    "tl_gemv_bf16_pf": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                c_float, c_int, c_void_p, c_size_t, c_void_p]),
    "tl_rope_table": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "tl_rope_kv_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_float, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "tl_attn_prefill_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                    c_int, c_int, c_int, c_float, c_void_p]),
    "tl_attn_decode_ws": (c_size_t, [c_int, c_int, c_int, c_int]),
    "tl_attn_decode_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int,
                                   c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "tl_attn_decode_fused": (c_int, [c_void_p] * 9 + [c_float, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "tl_decode_chain_ws": (c_size_t, [c_int, c_int, c_int, c_int]),
    "tl_decode_chain_trace": (c_int, [c_void_p, c_int]),
    "tl_decode_chain": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p, c_size_t, c_void_p]),
    "tl_peer_alloc": (c_int, [c_size_t, POINTER(c_void_p), c_void_p]),
    "tl_peer_open": (c_int, [c_void_p, POINTER(c_void_p)]),
    "tl_peer_close": (c_int, [c_void_p]),
    "tl_peer_free": (c_int, [c_void_p]),
    "tl_peer_wait": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, ctypes.c_uint64, c_void_p, c_void_p]),
    "tl_peer_signal": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "tl_peer_put": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p]),
    "tl_lmhead_ws": (c_size_t, [c_int, c_int]),
    "tl_lmhead_argmax": (c_int, [c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_size_t,
                                 c_int, c_int, c_int, c_void_p]),
    "tl_argmax_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_void_p]),
    "tl_sample_ws": (c_size_t, [c_int]),
    "tl_sample": (c_int, [c_void_p, c_void_p, c_int, c_int, c_float, c_int, c_float, ctypes.c_uint64, c_void_p, c_void_p, c_size_t,
                          c_void_p]),
    "tl_advance_pos": (c_int, [c_void_p, c_void_p, c_int, c_void_p]),
    "tl_append_token": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "tl_swiglu_fwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "tl_swiglu_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "tl_rmsnorm_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                               c_void_p]),
    "tl_rope_kv_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                               c_int, c_int, c_void_p]),
    "tl_qk_norm_bwd": (c_int, [c_void_p] * 6 + [c_float, c_int, c_int, c_int, c_int, c_void_p]),
    "tl_attn_bwd_ws": (c_size_t, [c_int, c_int, c_int]),
    "tl_attn_bwd": (c_int, [c_void_p] * 10 + [c_size_t, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "tl_ce_fwd_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_int, c_int, c_void_p]),
    "tl_embed_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "tl_colsum": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "tl_f32_to_bf16_accum": (c_int, [c_void_p, c_void_p, c_size_t, c_int, c_void_p]),
    "tl_add_inplace": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
    "tl_scale_add_bf16": (c_int, [c_void_p, c_void_p, c_float, c_int, c_size_t, c_void_p]),
    "tl_scale_add_f32": (c_int, [c_void_p, c_void_p, c_float, c_int, c_size_t, c_void_p]),
    "tl_adamw_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_float, c_float, c_float, c_float,
                              c_float, c_int, c_int, c_void_p]),
}



class DecodeJob(ctypes.Structure):
    """``tl_decode_job`` (include/tensorlink_b200.h)."""
    _fields_ = [("type", c_int32), ("N", c_int32), ("K", c_int32), ("flags", c_int32),
                ("n_h", c_int32), ("n_kv", c_int32), ("d", c_int32), ("T_max", c_int32),
                ("eps", c_float), ("scale", c_float),
                ("W", c_void_p), ("x", c_void_p), ("y", c_void_p), ("bias", c_void_p), ("residual", c_void_p),
                ("norm_w", c_void_p), ("pos_dev", c_void_p), ("cos_tab", c_void_p), ("sin_tab", c_void_p),
                ("q_norm_w", c_void_p), ("k_norm_w", c_void_p), ("k_cache", c_void_p), ("v_cache", c_void_p)]


JOB_GEMV, JOB_ATTN = 0, 1
ATTN_POS_PER_ROW = 1
CHAIN_MAX_JOBS, CHAIN_SYNC_BYTES = 16, 1024

_lib: Optional[ctypes.CDLL] = None


def load() -> ctypes.CDLL:
    """Load the shared library and bind every declared symbol (no device needed for this)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(tensorlink_b200 has no CPU or eager fallback)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)       # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def exported_symbols():
    return sorted(_SIGS)


def last_error() -> str:
    return (load().tl_last_error() or b"").decode()


def _check(rc: int, what: str):
    if rc != 0:
        raise NativeError(f"{what} failed ({rc}): {last_error()}")


_device_ok = False


def require_device():
    """Raise unless a B200-class (sm_100) device is current."""
    global _device_ok
    if _device_ok:
        return
    if not torch.cuda.is_available():
        raise NativeError("no CUDA device: the tensorlink_b200 shard executor runs on sm_100a only")
    sm, ma, mi = c_int(), c_int(), c_int()
    _check(load().tl_device_info(sm, ma, mi), "tl_device_info")
    _device_ok = True


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None:
        return None
    assert t.is_cuda, "device tensor expected"
    return t.data_ptr()


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream() -> int:
    """The current CUDA stream of the current device as a raw handle (every launch asks: the C accessor costs ~0.1 us,
    ``torch.cuda.current_stream().cuda_stream`` builds a Python Stream object each time)."""
    if _raw_stream is not None:
        return _raw_stream(torch.cuda.current_device())
    return torch.cuda.current_stream().cuda_stream


def _bf16(*ts):
    for t in ts:
        if t is not None:
            assert t.dtype == torch.bfloat16 and t.is_contiguous(), (t.dtype, t.is_contiguous())


# ------------------------------------------------------------------------------------------ thin typed wrappers
def rmsnorm_fwd(x: torch.Tensor, w: torch.Tensor, eps: float, out: Optional[torch.Tensor] = None,
                rstd: Optional[torch.Tensor] = None) -> torch.Tensor:
    require_device()
    _bf16(x, w, out)
    H = x.shape[-1]
    rows = x.numel() // H
    out = torch.empty_like(x) if out is None else out
    _check(load().tl_rmsnorm_fwd(_p(x), _p(w), _p(out), _p(rstd), rows, H, eps, _stream()), "tl_rmsnorm_fwd")
    return out


def embed_fwd(ids: torch.Tensor, table: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    require_device()
    assert ids.dtype == torch.int64 and ids.is_contiguous()
    _bf16(table, out)
    V, H = table.shape
    n = ids.numel()
    out = torch.empty(*ids.shape, H, dtype=torch.bfloat16, device=table.device) if out is None else out
    _check(load().tl_embed_fwd(_p(ids), _p(table), _p(out), n, H, V, _stream()), "tl_embed_fwd")
    return out


def gemm_splitk_ws(M: int, N: int) -> int:
    return int(load().tl_gemm_splitk_ws(M, N))


def gemm(a: torch.Tensor, b: torch.Tensor, out: Optional[torch.Tensor] = None, *, bias=None, residual=None,
         flags: int = 0, M: Optional[int] = None, N: Optional[int] = None, K: Optional[int] = None,
         ws: Optional[torch.Tensor] = None, norm_w: Optional[torch.Tensor] = None, eps: float = 1e-6,
         h_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """C[M,N] = A·B^T with the epilogue ``flags``.  A is [M,K] (or [K,M] with A_MN_MAJOR), B is [N,K] (or [K,N])."""
    require_device()
    _bf16(a, b, bias, residual)
    a_mn, b_mn = bool(flags & A_MN_MAJOR), bool(flags & B_MN_MAJOR)
    if M is None:
        M = a.shape[1] if a_mn else a.shape[0]
    if K is None:
        K = a.shape[0] if a_mn else a.shape[1]
    if N is None:
        N = b.shape[1] if b_mn else b.shape[0]
    c_cols = N // 2 if flags & EPI_SWIGLU else N
    if out is None:
        out = torch.empty(M, c_cols, dtype=torch.float32 if flags & EPI_OUT_F32 else torch.bfloat16, device=a.device)
    if bias is not None:
        flags |= EPI_BIAS
    if residual is not None:
        flags |= EPI_RESIDUAL
    if norm_w is not None:          # also h_out = RMSNorm(out) * norm_w (fused into the split-K reduce when that path runs)
        assert h_out is not None and h_out.dtype == torch.bfloat16 and h_out.is_contiguous() and h_out.shape == out.shape
        _check(load().tl_gemm_bf16_ws_norm(_p(a), _p(b), _p(out), M, N, K, a.stride(0), b.stride(0), out.stride(0), _p(bias),
                                           _p(residual), flags, _p(ws), 0 if ws is None else ws.numel() * ws.element_size(),
                                           _p(norm_w), eps, _p(h_out), _stream()), "tl_gemm_bf16_ws_norm")
        return out
    if ws is not None:
        _check(load().tl_gemm_bf16_ws(_p(a), _p(b), _p(out), M, N, K, a.stride(0), b.stride(0), out.stride(0), _p(bias),
                                      _p(residual), flags, _p(ws), ws.numel() * ws.element_size(), _stream()),
               "tl_gemm_bf16_ws")
        return out
    _check(load().tl_gemm_bf16(_p(a), _p(b), _p(out), M, N, K, a.stride(0), b.stride(0), out.stride(0), _p(bias),
                               _p(residual), flags, _stream()), "tl_gemm_bf16")
    return out


_PREFETCH_BYTES = None


def prefetch_bytes() -> int:
    """How much of the next launch's weights a GEMV asks L2 to fetch (TL_PREFETCH_MB, default 8 — measured best of 0/8/32/64: 349.0 / 355.6 / 352.1 / 351.7 tok/s; 0 disables)."""
    global _PREFETCH_BYTES
    if _PREFETCH_BYTES is None:
        _PREFETCH_BYTES = int(float(os.environ.get("TL_PREFETCH_MB", "8")) * (1 << 20))
    return _PREFETCH_BYTES


def gemv(x: torch.Tensor, w: torch.Tensor, out: Optional[torch.Tensor] = None, *, bias=None, residual=None,
         norm_w=None, eps: float = 1e-6, flags: int = 0, next_w: Optional[torch.Tensor] = None) -> torch.Tensor:
    require_device()
    _bf16(x, w, bias, residual, norm_w, out)
    M, K = x.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty(M, N // 2 if flags & EPI_SWIGLU else N, dtype=torch.bfloat16, device=x.device)
    if bias is not None:
        flags |= EPI_BIAS
    if residual is not None:
        flags |= EPI_RESIDUAL
    if next_w is not None and prefetch_bytes() > 0:
        nb = min(next_w.numel() * next_w.element_size(), prefetch_bytes())
        _check(load().tl_gemv_bf16_pf(_p(x), _p(w), _p(out), M, N, K, _p(bias), _p(residual), _p(norm_w), eps, flags,
                                      _p(next_w), nb, _stream()), "tl_gemv_bf16_pf")
        return out
    _check(load().tl_gemv_bf16(_p(x), _p(w), _p(out), M, N, K, _p(bias), _p(residual), _p(norm_w), eps, flags,
                               _stream()), "tl_gemv_bf16")
    return out


def rope_table(inv_freq: torch.Tensor, max_pos: int):
    require_device()
    assert inv_freq.dtype == torch.float32 and inv_freq.is_cuda
    half = inv_freq.numel()
    cos = torch.empty(max_pos, half, dtype=torch.bfloat16, device=inv_freq.device)
    sin = torch.empty_like(cos)
    _check(load().tl_rope_table(_p(inv_freq), _p(cos), _p(sin), max_pos, half, _stream()), "tl_rope_table")
    return cos, sin


def rope_kv_fwd(qkv, q_out, k_cache, v_cache, pos0_dev, cos_tab, sin_tab, q_norm_w, k_norm_w, eps, S, n_h, n_kv, d):
    require_device()
    _bf16(qkv, q_out, k_cache, v_cache, cos_tab, sin_tab, q_norm_w, k_norm_w)
    n_tokens = qkv.shape[0]
    T_max = k_cache.shape[2]
    _check(load().tl_rope_kv_fwd(_p(qkv), _p(q_out), _p(k_cache), _p(v_cache), _p(pos0_dev), _p(cos_tab), _p(sin_tab),
                                 _p(q_norm_w), _p(k_norm_w), eps, n_tokens, S, n_h, n_kv, d, T_max, _stream()),
           "tl_rope_kv_fwd")


def attn_prefill_fwd(q, k_cache, v_cache, out, lse, B, S, past_len, n_h, n_kv, d, scale):
    require_device()
    _bf16(q, k_cache, v_cache, out)
    T_max = k_cache.shape[2]
    _check(load().tl_attn_prefill_fwd(_p(q), _p(k_cache), _p(v_cache), _p(out), _p(lse), B, S, past_len, n_h, n_kv, d,
                                      T_max, scale, _stream()), "tl_attn_prefill_fwd")


def attn_decode_ws(B, n_h, d, T_max) -> int:
    return int(load().tl_attn_decode_ws(B, n_h, d, T_max))


def attn_decode_fwd(q, k_cache, v_cache, out, kv_len_dev, ws, B, n_h, n_kv, d, scale):
    require_device()
    _bf16(q, k_cache, v_cache, out)
    T_max = k_cache.shape[2]
    _check(load().tl_attn_decode_fwd(_p(q), _p(k_cache), _p(v_cache), _p(out), _p(kv_len_dev), _p(ws),
                                     ws.numel() * ws.element_size(), B, n_h, n_kv, d, T_max, scale, _stream()),
           "tl_attn_decode_fwd")


def lmhead_ws(M, V) -> int:
    return int(load().tl_lmhead_ws(M, V))


def lmhead_argmax(x, w, norm_w, eps, ids_out, logits_out, ws):
    require_device()
    _bf16(x, w, norm_w, logits_out)
    M, H = x.shape
    V = w.shape[0]
    assert ids_out.dtype == torch.int64
    _check(load().tl_lmhead_argmax(_p(x), _p(w), _p(norm_w), eps, _p(ids_out), _p(logits_out), _p(ws),
                                   ws.numel() * ws.element_size(), M, V, H, _stream()), "tl_lmhead_argmax")


def argmax_bf16(logits, ids_out, ws):
    require_device()
    _bf16(logits)
    M, V = logits.shape
    _check(load().tl_argmax_bf16(_p(logits), _p(ids_out), _p(ws), ws.numel() * ws.element_size(), M, V, _stream()),
           "tl_argmax_bf16")


def sample_ws(M: int) -> int:
    return int(load().tl_sample_ws(M))


def sample(logits, ids_out, counters, ws, temperature: float = 1.0, top_k: int = 0, top_p: float = 1.0, seed: int = 0):
    """ids_out[m] ~ softmax(top-p(top-k(logits[m] / temperature))); ``counters`` int32[M] advance by one per call."""
    require_device()
    _bf16(logits)
    M, V = logits.shape
    assert ids_out.dtype == torch.int64 and counters.dtype == torch.int32 and counters.numel() >= M
    _check(load().tl_sample(_p(logits), _p(ids_out), M, V, float(temperature), int(top_k or 0), float(top_p), int(seed) & (2 ** 64 - 1),
                            _p(counters), _p(ws), ws.numel() * ws.element_size(), _stream()), "tl_sample")


def advance_pos(pos_dev, kv_len_dev, delta: int):
    require_device()
    _check(load().tl_advance_pos(_p(pos_dev), _p(kv_len_dev), delta, _stream()), "tl_advance_pos")


def append_token(ids, out_tokens, step_dev):
    require_device()
    assert ids.dtype == torch.int64 and out_tokens.dtype == torch.int64 and out_tokens.is_contiguous()
    B, ld = out_tokens.shape
    _check(load().tl_append_token(_p(ids), _p(out_tokens), _p(step_dev), B, ld, _stream()), "tl_append_token")


# ------------------------------------------------------------------------------------------ peer-memory mailboxes
class _RawCuda:
    """A raw device allocation seen through ``__cuda_array_interface__`` (bytes), so torch can view it."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3,
                                         "strides": None}


def tensor_from_ptr(ptr: int, nbytes: int) -> torch.Tensor:
    """uint8 tensor over [ptr, ptr+nbytes) without taking ownership (the caller keeps the allocation alive).
    No target device is named: torch tags the view with the device that owns the memory (for a peer mapping, the
    neighbour's), and naming another one would silently turn the view into a copy.  Only ``data_ptr()`` of such a
    view is ever used (as a kernel argument); torch never launches work on it."""
    return torch.as_tensor(_RawCuda(ptr, nbytes))


def peer_alloc(nbytes: int):
    """(ptr, handle bytes[64]): zeroed device allocation exportable to other processes on this node."""
    require_device()
    ptr, h = c_void_p(), ctypes.create_string_buffer(64)
    _check(load().tl_peer_alloc(nbytes, ctypes.byref(ptr), h), "tl_peer_alloc")
    return ptr.value, bytes(h.raw)


def peer_open(handle: bytes) -> int:
    require_device()
    ptr = c_void_p()
    _check(load().tl_peer_open(ctypes.create_string_buffer(handle, 64), ctypes.byref(ptr)), "tl_peer_open")
    return ptr.value


def peer_close(ptr: int):
    _check(load().tl_peer_close(ptr), "tl_peer_close")


def peer_free(ptr: int):
    _check(load().tl_peer_free(ptr), "tl_peer_free")


def peer_wait(flag, want, err, wait_ns=None, timeout_ns: int = 0, bump=None):
    require_device()
    _check(load().tl_peer_wait(_p(flag), _p(want), _p(err), _p(wait_ns), timeout_ns, _p(bump), _stream()), "tl_peer_wait")


def peer_signal(flag_peer, sent, bump=None):
    require_device()
    _check(load().tl_peer_signal(_p(flag_peer), _p(sent), _p(bump), _stream()), "tl_peer_signal")


def peer_put(dst_peer, src, flag_peer, sent):
    require_device()
    nbytes = src.numel() * src.element_size()
    _check(load().tl_peer_put(_p(dst_peer), _p(src), nbytes, _p(flag_peer), _p(sent), _stream()), "tl_peer_put")


# ------------------------------------------------------------------------------------------ training wrappers
def swiglu_fwd(gu, h):
    require_device(); _bf16(gu, h)
    M, I = h.shape
    _check(load().tl_swiglu_fwd(_p(gu), _p(h), M, I, _stream()), "tl_swiglu_fwd")


def swiglu_bwd(gu, dh, dgu):
    require_device(); _bf16(gu, dh, dgu)
    M, I = dh.shape
    _check(load().tl_swiglu_bwd(_p(gu), _p(dh), _p(dgu), M, I, _stream()), "tl_swiglu_bwd")


def rmsnorm_bwd(x, w, dy, rstd, dx, dw_accum, dx_add=None):
    require_device(); _bf16(x, w, dy, dx, dx_add)
    H = x.shape[-1]
    _check(load().tl_rmsnorm_bwd(_p(x), _p(w), _p(dy), _p(rstd), _p(dx_add), _p(dx), _p(dw_accum), x.numel() // H, H,
                                 _stream()), "tl_rmsnorm_bwd")


def rope_kv_bwd(dq, dk, dv, dqkv, cos_tab, sin_tab, S, n_h, n_kv, d):
    # the kernel takes T_max from dk and indexes every buffer from these sizes: a mismatch would read or write out of bounds
    n_tokens = dqkv.shape[0]
    assert n_tokens % S == 0 and tuple(dqkv.shape) == (n_tokens, (n_h + 2 * n_kv) * d), (tuple(dqkv.shape), S, n_h, n_kv, d)
    assert dq.numel() == n_tokens * n_h * d, (tuple(dq.shape), n_tokens, n_h, d)
    assert tuple(dk.shape) == tuple(dv.shape) == (n_tokens // S, n_h, dk.shape[2], d) and dk.shape[2] >= S, \
        (tuple(dk.shape), tuple(dv.shape), S, n_h, d)
    assert cos_tab.shape == sin_tab.shape and cos_tab.shape[0] >= S and cos_tab.shape[1] == d // 2, (tuple(cos_tab.shape), S, d)
    require_device(); _bf16(dq, dk, dv, dqkv)
    _check(load().tl_rope_kv_bwd(_p(dq), _p(dk), _p(dv), _p(dqkv), _p(cos_tab), _p(sin_tab), dqkv.shape[0], S, n_h, n_kv,
                                 d, dk.shape[2], _stream()), "tl_rope_kv_bwd")


def attn_bwd_ws(B, S, n_h) -> int:
    return int(load().tl_attn_bwd_ws(B, S, n_h))


def attn_bwd(q, k_cache, v_cache, out, dout, lse, dq, dk, dv, ws, B, S, n_h, n_kv, d, scale):
    # T_max comes from k_cache and is also the row pitch of dk / dv: their shapes must agree with it
    T_max = k_cache.shape[2]
    assert tuple(k_cache.shape) == tuple(v_cache.shape) == (B, n_kv, T_max, d) and S <= T_max, \
        (tuple(k_cache.shape), tuple(v_cache.shape), B, S, n_kv, d)
    assert tuple(dk.shape) == tuple(dv.shape) == (B, n_h, T_max, d), (tuple(dk.shape), tuple(dv.shape), B, n_h, T_max, d)
    n = B * S * n_h * d
    assert q.numel() == out.numel() == dout.numel() == dq.numel() == n and lse.numel() == B * n_h * S, \
        (tuple(q.shape), tuple(out.shape), tuple(dout.shape), tuple(dq.shape), tuple(lse.shape), B, S, n_h, d)
    require_device(); _bf16(q, k_cache, v_cache, out, dout, dq, dk, dv)
    _check(load().tl_attn_bwd(_p(q), _p(k_cache), _p(v_cache), _p(out), _p(dout), _p(lse), _p(dq), _p(dk), _p(dv), _p(ws),
                              ws.numel() * ws.element_size(), B, S, n_h, n_kv, d, T_max, scale, _stream()),
           "tl_attn_bwd")


def ce_fwd_bwd(logits, labels, loss_sum, n_valid, dlogits, grad_scale: float):
    require_device(); _bf16(logits, dlogits)
    M, V = logits.shape
    assert labels.dtype == torch.int64 and loss_sum.dtype == torch.float32
    _check(load().tl_ce_fwd_bwd(_p(logits), _p(labels), _p(loss_sum), _p(n_valid), _p(dlogits), grad_scale, M, V,
                                _stream()), "tl_ce_fwd_bwd")


def embed_bwd(ids, dout, dtable):
    """dtable[id] += the fp32 sum of dout's rows of the tokens holding id, rounded once (deterministic); ids outside
    [0, V) are skipped."""
    V, H = dtable.shape
    n = ids.numel()
    assert ids.dtype == torch.int64, ids.dtype
    assert dout.shape[-1] == H and dout.numel() == n * H, (tuple(dout.shape), n, H)
    require_device(); _bf16(dout, dtable)
    sorted_ids, order = torch.sort(ids.reshape(-1), stable=True)     # one run per distinct id, tokens in order
    _check(load().tl_embed_bwd(_p(sorted_ids), _p(order), _p(dout), _p(dtable), n, H, V, _stream()), "tl_embed_bwd")


def colsum(dy, db_accum):
    require_device()
    assert db_accum.dtype == torch.float32
    M, N = dy.shape
    _check(load().tl_colsum(_p(dy), _p(db_accum), M, N, dy.stride(0), _stream()), "tl_colsum")


def f32_to_bf16_accum(src, dst, accumulate: bool):
    require_device()
    _check(load().tl_f32_to_bf16_accum(_p(src), _p(dst), src.numel(), int(accumulate), _stream()), "tl_f32_to_bf16_accum")


def add_inplace(a, b):
    require_device(); _bf16(a, b)
    _check(load().tl_add_inplace(_p(a), _p(b), a.numel(), _stream()), "tl_add_inplace")


def scale_add(a, b, scale: float, accumulate: bool = True):
    """a = (a if accumulate else 0) + scale * b   (bf16 or fp32 pairs, same shape)."""
    require_device()
    assert a.dtype == b.dtype and a.numel() == b.numel() and a.is_contiguous() and b.is_contiguous()
    if a.dtype == torch.bfloat16:
        _check(load().tl_scale_add_bf16(_p(a), _p(b), scale, int(accumulate), a.numel(), _stream()), "tl_scale_add_bf16")
    else:
        assert a.dtype == torch.float32
        _check(load().tl_scale_add_f32(_p(a), _p(b), scale, int(accumulate), a.numel(), _stream()), "tl_scale_add_f32")


def adamw_step(param, grad, m, v, lr, beta1, beta2, eps, wd, step: int, decoupled: bool):
    require_device()
    _check(load().tl_adamw_step(_p(param), _p(grad), _p(m), _p(v), param.numel(), lr, beta1, beta2, eps, wd, step,
                                int(decoupled), _stream()), "tl_adamw_step")


def attn_decode_fused(qkv, k_cache, v_cache, out, pos_dev, cos_tab, sin_tab, q_norm_w, k_norm_w, eps, B, n_h, n_kv, d, scale):
    require_device(); _bf16(qkv, k_cache, v_cache, out)
    _check(load().tl_attn_decode_fused(_p(qkv), _p(k_cache), _p(v_cache), _p(out), _p(pos_dev), _p(cos_tab), _p(sin_tab),
                                       _p(q_norm_w), _p(k_norm_w), eps, B, n_h, n_kv, d, k_cache.shape[2], scale, _stream()),
           "tl_attn_decode_fused")


def decode_chain_ws(M: int, n_h: int, n_kv: int, d: int) -> int:
    return int(load().tl_decode_chain_ws(M, n_h, n_kv, d))


CHAIN_TRACE_WORDS = 2 * (CHAIN_MAX_JOBS + 1) * 4 + CHAIN_MAX_JOBS * 160 + CHAIN_MAX_JOBS * 4


def decode_chain_trace(buf: Optional[torch.Tensor]):
    """``buf``: int64 [n_slots, CHAIN_TRACE_WORDS] (or None to switch tracing off)."""
    _check(load().tl_decode_chain_trace(_p(buf), 0 if buf is None else buf.shape[0]), "tl_decode_chain_trace")


def make_job(type_, **kw) -> DecodeJob:
    j = DecodeJob()
    j.type = type_
    for k, v in kw.items():
        if isinstance(v, torch.Tensor):
            v = v.data_ptr()
        setattr(j, k, v)
    return j


class DecodeChain:
    """One launch site of ``tl_decode_chain``: a host job array (kept alive here: a captured graph holds the parameter
    copy, eager launches re-read this array), the rows per step, the private sync slot and the prefetch hint."""

    def __init__(self, jobs, M: int, sync_slot: torch.Tensor, attn_ws: torch.Tensor, next_w: Optional[torch.Tensor] = None):
        assert 1 <= len(jobs) <= CHAIN_MAX_JOBS
        self.n, self.M = len(jobs), M
        self.host = (DecodeJob * self.n)(*jobs)
        self.sync_slot, self.attn_ws, self.next_w = sync_slot, attn_ws, next_w
        assert sync_slot.numel() * sync_slot.element_size() >= CHAIN_SYNC_BYTES

    def launch(self):
        require_device()
        nb = 0
        if self.next_w is not None and prefetch_bytes() > 0:
            nb = min(self.next_w.numel() * self.next_w.element_size(), prefetch_bytes())
        _check(load().tl_decode_chain(ctypes.cast(self.host, c_void_p), self.n, self.M, _p(self.sync_slot), _p(self.attn_ws),
                                      self.attn_ws.numel() * self.attn_ws.element_size(), _p(self.next_w) if nb else None, nb,
                                      _stream()), "tl_decode_chain")


def qk_norm_bwd(qkv_pre, dqkv, qn, kn, dqn_acc, dkn_acc, eps, n_h, n_kv, d):
    require_device(); _bf16(qkv_pre, dqkv, qn, kn)
    _check(load().tl_qk_norm_bwd(_p(qkv_pre), _p(dqkv), _p(qn), _p(kn), _p(dqn_acc), _p(dkn_acc), eps, dqkv.shape[0], n_h,
                                 n_kv, d, _stream()), "tl_qk_norm_bwd")
