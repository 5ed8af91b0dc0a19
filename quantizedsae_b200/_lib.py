"""ctypes binding of libqsae_b200.so (C ABI: include/qsae_b200.h).

There is no fallback: if the library is missing it is built with nvcc, and if that fails, or a
call returns a non-zero status, a QsaeError is raised. torch is used only to own device memory
and to supply the current CUDA stream.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import torch

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libqsae_b200.so"

QSAE_MAX_K = 224
QSAE_MAX_K_LARGE = 4096
QSAE_RESCORE_MARGIN = 16
ACT_NONE, ACT_RELU = 0, 1

# every symbol include/qsae_b200.h declares: name -> (restype, argtypes)
_vp, _i, _f, _sz = C.c_void_p, C.c_int, C.c_float, C.c_size_t
SYMBOLS = {
    "qsae_abi_version": (_i, []),
    "qsae_last_error": (C.c_char_p, []),
    "qsae_check_device": (_i, []),
    "qsae_cast_f32_to_bf16": (_i, [_vp, _vp, _sz, _vp]),
    "qsae_pack_bitplanes": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp]),
    "qsae_dequant_soft": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "qsae_transpose_f32": (_i, [_vp, _i, _i, _vp, _vp]),
    "qsae_encode_topk_workspace_bytes": (_i, [_i, _i, _i, _i, _i, C.POINTER(_sz)]),
    "qsae_prepare_encoder_sample": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "qsae_set_encode_kernel_events": (_i, [_vp, _vp]),
    "qsae_launch_count": (C.c_ulonglong, []),
    "qsae_reload_tuning": (_i, []),
    "qsae_default_sample_rows": (_i, [_i]),
    "qsae_set_stage_events": (_i, [_vp, _i]),
    "qsae_set_unordered_topk": (_i, [_i]),
    "qsae_prior_prep": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, C.POINTER(_i), _vp]),
    "qsae_encode_topk": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "qsae_bsae_forward": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _i, _f, _vp, _vp, _vp, _vp, _vp, _vp,
                               _sz, _vp]),
    "qsae_encode_dense_tc": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "qsae_encode_dense_f32": (_i, [_vp, _vp, _i, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "qsae_topk_dense_workspace_bytes": (_i, [_i, _i, _i, C.POINTER(_sz)]),
    "qsae_topk_dense": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "qsae_decode_int4": (_i, [_vp, _vp, _i, _i, _vp, _i, _i, _f, _vp, _vp, _vp]),
    "qsae_decode_int8": (_i, [_vp, _vp, _i, _i, _vp, _i, _i, _f, _vp, _vp, _vp]),
    "qsae_decode_rows_f32": (_i, [_vp, _vp, _i, _i, _vp, _i, _i, _f, _vp, _vp, _vp]),
    "qsae_pack_matryoshka": (_i, [_vp, _vp, _i, _i, _vp, _vp, _i, _vp, _vp, _vp]),
    "qsae_matryoshka_workspace_bytes": (_i, [_i, _i, _i, C.POINTER(_sz)]),
    "qsae_matryoshka_forward": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "qsae_matryoshka_forward_active": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _i, _i, _vp, _vp, _vp,
                                            _vp, _i, _vp, _vp, _vp, _sz, _vp]),
    "qsae_activation_counts": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "qsae_coactivation": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "qsae_coactivation_dense": (_i, [_vp, _i, _i, _vp, _vp, _vp]),
    "qsae_sq_error_accumulate": (_i, [_vp, _vp, _sz, _vp, _vp]),
    "qsae_compact_dense": (_i, [_vp, _i, _i, _i, _f, _i, _vp, _vp, _vp, _vp, _vp]),
    "qsae_max_row_norm": (_i, [_vp, _i, _i, _vp, _vp]),
    "qsae_residual_update": (_i, [_vp, _vp, _sz, _vp, _vp]),
    "qsae_unpack_matryoshka_t": (_i, [_vp, _i, _i, _vp, _vp]),
    "qsae_matryoshka_dense_workspace_bytes": (_i, [_i, _i, _i, C.POINTER(_sz)]),
    "qsae_matryoshka_forward_dense": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(_i), _i, _vp, _i, _i, _i, _vp,
                                           _vp, _vp, _sz, _vp]),
    "qsae_matryoshka_forward_dense_active": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(_i), _i, _vp, _i, _i, _i,
                                                  _vp, _vp, _vp, _i, _i, _vp, _sz, _vp]),
    "qsae_decode_matryoshka_lists_workspace_bytes": (_i, [C.POINTER(_sz)]),
    "qsae_decode_matryoshka_lists": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "qsae_pack_ternary": (_i, [_vp, _i, _i, _f, _vp, _vp, _vp]),
    "qsae_split_bf16": (_i, [_vp, _vp, _vp, _sz, _vp]),
    "qsae_decode_dense_workspace_bytes": (_i, [_i, _i, _i, C.POINTER(_sz)]),
    "qsae_decode_dense": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "qsae_tsae_workspace_bytes": (_i, [_i, _i, _i, _i, C.POINTER(_sz)]),
    "qsae_split_bf16x3": (_i, [_vp, _vp, _vp, _vp, _sz, _vp]),
    "qsae_tsae_forward": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "qsae_pack_candidates": (_i, [_vp, _vp, _sz, _vp, _vp]),
    "qsae_merge_candidates_workspace_bytes": (_i, [_i, C.POINTER(_sz)]),
    "qsae_merge_candidates": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "qsae_peer_alloc": (_i, [_sz, C.POINTER(_vp)]),
    "qsae_peer_free": (_i, [_vp]),
    "qsae_peer_export": (_i, [_vp, C.c_char_p]),
    "qsae_peer_import": (_i, [C.c_char_p, C.POINTER(_vp)]),
    "qsae_peer_close": (_i, [_vp]),
    "qsae_peer_signal": (_i, [_vp, _i, C.c_uint, _vp]),
    "qsae_peer_wait": (_i, [_vp, _i, C.c_uint, _vp, _vp]),
    "qsae_merge_candidates_peer": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "qsae_reduce_partials_peer": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "qsae_decode_int4_range": (_i, [_vp, _vp, _i, _i, _vp, _i, _i, _i, _f, _vp, _vp, _vp]),
    "qsae_decode_int8_range": (_i, [_vp, _vp, _i, _i, _vp, _i, _i, _i, _f, _vp, _vp, _vp]),
    "qsae_decode_rows_f32_range": (_i, [_vp, _vp, _i, _i, _vp, _i, _i, _i, _f, _vp, _vp, _vp]),
    "qsae_densify": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "qsae_bsae_plan_create": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _f, _i, _i, C.POINTER(_vp)]),
    "qsae_bsae_plan_destroy": (None, [_vp]),
    "qsae_bsae_forward_host": (_i, [_vp, _vp, _i, _vp, _vp, _vp]),
    "qsae_bsae_submit_host": (_i, [_vp, _vp, _i, _vp, _vp, _vp, C.POINTER(_i)]),
    "qsae_bsae_wait_host": (_i, [_vp, _i]),
    "qsae_bsae_plan_set_io": (_i, [_vp, _i, _i]),
    "qsae_rows_scatter_add": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _f, _vp, _vp, _vp]),
    "qsae_rows_gather_dot": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _f, _vp, _vp]),
    "qsae_column_sum": (_i, [_vp, _i, _i, _f, _vp, _vp]),
    "qsae_bsae_logit_grad": (_i, [_vp, _vp, _i, _i, _i, _vp, _f, _i, _vp, _vp]),
    "qsae_matryoshka_backward_scatter": (_i, [_vp, _i, _i, _i, _i, C.POINTER(_vp), C.POINTER(_i), _i, _vp, _vp, _vp]),
    "qsae_matryoshka_backward_finish": (_i, [_vp, _vp, _vp, _vp, _vp, C.POINTER(_i), _i, _i, _i, _f, _i, _vp, _vp, _vp]),
    "qsae_matryoshka_backward_dense_workspace_bytes": (_i, [_i, _i, _i, _i, C.POINTER(_sz)]),
    "qsae_matryoshka_backward_dense": (_i, [_vp, _i, _i, _i, C.POINTER(_vp), C.POINTER(_i), _i, _vp, _vp, _vp, _i, _vp, _vp, _vp,
                                            _vp, _sz, _vp]),
    "qsae_rigl_workspace_bytes": (_i, [C.POINTER(_sz)]),
    "qsae_rigl_init_mask": (_i, [_vp, _vp, _i, _i, C.c_ulonglong, _vp, _sz, _vp]),
    "qsae_rigl_update_mask": (_i, [_vp, _vp, _vp, _vp, _i, _i, C.c_ulonglong, C.c_ulonglong, _vp, _sz, _vp]),
    "qsae_mul_inplace": (_i, [_vp, _vp, _sz, _vp]),
    "qsae_pack_ternary_t": (_i, [_vp, _i, _i, _f, _vp, _vp]),
    "qsae_wgrad": (_i, [C.POINTER(_vp), C.POINTER(_vp), _i, _i, _i, _i, _i, _vp, _vp]),
    "qsae_tsae_backward_workspace_bytes": (_i, [_i, _i, _i, _i, C.POINTER(_sz)]),
    "qsae_tsae_backward": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "qsae_baseline_backward_workspace_bytes": (_i, [_i, _i, _i, _i, C.POINTER(_sz)]),
    "qsae_baseline_backward": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz,
                                    _vp]),
    "qsae_baseline_backward_range_workspace_bytes": (_i, [_i, _i, _i, _i, C.POINTER(_sz)]),
    "qsae_baseline_backward_range": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "qsae_bsae_backward_workspace_bytes": (_i, [_i, _i, _i, _i, _i, C.POINTER(_sz)]),
    "qsae_bsae_backward": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _f, _vp, _f, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp,
                                _sz, _vp]),
}


class QsaeError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"libqsae_b200 status {status}: {message}")
        self.status = status


_lib = None


def launch_count() -> int:
    """Kernels libqsae_b200.so has launched in this process (counted in C: qsae_launch_count)."""
    return int(load().qsae_launch_count())


def load(build_if_missing: bool = True) -> C.CDLL:
    """dlopen the library and type every symbol; raises if it cannot be loaded."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        if not build_if_missing:
            raise QsaeError(-100, f"{LIB_PATH} is missing (run python -m quantizedsae_b200.build)")
        from . import build as _build

        _build.build()
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    if lib.qsae_abi_version() != 1:
        raise QsaeError(-101, "ABI version mismatch between _lib.py and libqsae_b200.so")
    _lib = lib
    return lib


def check(status: int) -> None:
    if status != 0:
        msg = load().qsae_last_error().decode(errors="replace")
        if status == -5:
            raise RuntimeError(msg)  # torch.topk raises RuntimeError for k > H as well
        raise QsaeError(status, msg)


class unordered_topk:
    """Context manager: large fast-mode selections (k > QSAE_MAX_K, candidate merges) inside the block return their
    winners as a set, in no particular order (qsae_set_unordered_topk)."""

    def __init__(self, on: bool = True):
        self.on = bool(on)

    def __enter__(self):
        if self.on:
            check(load().qsae_set_unordered_topk(1))
        return self

    def __exit__(self, *exc):
        if self.on:
            check(load().qsae_set_unordered_topk(0))
        return False


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: torch.Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


def _need_cuda(*ts: torch.Tensor) -> None:
    for t in ts:
        if t is not None and not t.is_cuda:
            raise QsaeError(-102, "libqsae_b200 kernels need CUDA tensors; there is no CPU path")
        if t is not None and not t.is_contiguous():
            raise QsaeError(-103, "libqsae_b200 kernels need contiguous tensors")


# ------------------------------------------------------------------------------------------
# thin typed wrappers (allocate outputs with torch, launch on torch's current stream)
# ------------------------------------------------------------------------------------------

def cast_bf16(src: torch.Tensor) -> torch.Tensor:
    _need_cuda(src)
    assert src.dtype == torch.float32
    dst = torch.empty(src.shape, dtype=torch.bfloat16, device=src.device)
    check(load().qsae_cast_f32_to_bf16(src.data_ptr(), dst.data_ptr(), src.numel(), _stream()))
    return dst


def pack_bitplanes(logits: torch.Tensor, D: int, n_bits: int, want_stats: bool = True):
    """-> (packed uint8 [H, D/2] or int8-as-uint8 [H, D], polarize_loss float|None, max_gap float|None)."""
    _need_cuda(logits)
    H = logits.shape[0]
    assert logits.dtype == torch.float32 and logits.shape[1] == D * n_bits
    cols = D // 2 if n_bits <= 4 else D
    packed = torch.empty((H, cols), dtype=torch.uint8, device=logits.device)
    stats = torch.zeros(2, dtype=torch.float64, device=logits.device) if want_stats else None
    check(load().qsae_pack_bitplanes(logits.data_ptr(), H, D, n_bits, packed.data_ptr(), _ptr(stats), _stream()))
    if not want_stats:
        return packed, None, None
    s = stats.cpu()
    return packed, float(s[0]) / (H * D * n_bits), float(s[1])


def dequant_soft(logits: torch.Tensor, D: int, n_bits: int) -> torch.Tensor:
    _need_cuda(logits)
    H = logits.shape[0]
    rows = torch.empty((H, D), dtype=torch.float32, device=logits.device)
    check(load().qsae_dequant_soft(logits.data_ptr(), H, D, n_bits, rows.data_ptr(), _stream()))
    return rows


def transpose(src: torch.Tensor) -> torch.Tensor:
    _need_cuda(src)
    R, Cc = src.shape
    dst = torch.empty((Cc, R), dtype=torch.float32, device=src.device)
    check(load().qsae_transpose_f32(src.data_ptr(), R, Cc, dst.data_ptr(), _stream()))
    return dst


def encode_topk_workspace_bytes(B: int, H: int, D: int, k: int, n_sample: int = 0) -> int:
    n = _sz(0)
    check(load().qsae_encode_topk_workspace_bytes(B, H, D, k, n_sample, C.byref(n)))
    return int(n.value)


def default_sample_rows(H: int) -> int:
    """Rows of the sampled dictionary used for the prior threshold (0 = do not sample)."""
    return int(load().qsae_default_sample_rows(int(H)))


def prepare_sample(w_bf16: torch.Tensor, b_enc: torch.Tensor, n_sample: int | None = None):
    """-> (w_sample [n,D] bf16, b_sample [n] f32) or None when the dictionary is too small."""
    _need_cuda(w_bf16, b_enc)
    H, D = w_bf16.shape
    n = default_sample_rows(H) if n_sample is None else n_sample
    if n <= 0:
        return None
    ws = torch.empty((n, D), dtype=torch.bfloat16, device=w_bf16.device)
    bs = torch.empty((n,), dtype=torch.float32, device=w_bf16.device)
    check(load().qsae_prepare_encoder_sample(w_bf16.data_ptr(), b_enc.data_ptr(), H, D, n, ws.data_ptr(),
                                             bs.data_ptr(), _stream()))
    return ws, bs


def prior_prep(x: torch.Tensor, sample, m: int, act: int = ACT_NONE):
    """The single-launch cast + sample pre-pass + prior of the small-batch path -> (x_bf16 [B,D], prior [B], ns)."""
    w_s, b_s = sample
    _need_cuda(x, w_s, b_s)
    B, D = x.shape
    xb = torch.empty((B, D), dtype=torch.bfloat16, device=x.device)
    prior = torch.empty((B,), dtype=torch.float32, device=x.device)
    ns = _i(0)
    check(load().qsae_prior_prep(x.data_ptr(), w_s.data_ptr(), b_s.data_ptr(), w_s.shape[0], B, D, act, m,
                                 xb.data_ptr(), prior.data_ptr(), C.byref(ns), _stream()))
    return xb, prior, int(ns.value)


_ws_cache: dict = {}


_WS_ALIGN = 1024   # the TMA-fed kernels want 1024-byte aligned workspaces; torch's small-block pool gives 512


def _workspace(device, nbytes: int) -> torch.Tensor:
    """Per (device, stream) scratch buffer, grown on demand, 1024-byte aligned."""
    key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    ws = _ws_cache.get(key)
    if ws is None or ws.numel() < nbytes:
        raw = torch.empty(nbytes + _WS_ALIGN, dtype=torch.uint8, device=device)
        off = (-raw.data_ptr()) % _WS_ALIGN
        ws = raw[off:off + nbytes]
        _ws_cache[key] = ws
    return ws


def encode_topk(x: torch.Tensor, w_bf16: torch.Tensor, w_f32: torch.Tensor | None, b_enc: torch.Tensor,
                k: int, act: int = ACT_NONE, exact: bool = False, want_flags: bool = False, sample=None):
    """-> (vals [B,k] f32, idx [B,k] i32, flags [B] i32 | None)"""
    _need_cuda(x, w_bf16, w_f32, b_enc)
    B, D = x.shape
    H = w_bf16.shape[0]
    assert x.dtype == torch.float32 and w_bf16.dtype == torch.bfloat16 and b_enc.dtype == torch.float32
    vals = torch.empty((B, k), dtype=torch.float32, device=x.device)
    idx = torch.empty((B, k), dtype=torch.int32, device=x.device)
    flags = torch.empty((B,), dtype=torch.int32, device=x.device) if want_flags else None
    if B == 0:
        return vals, idx, flags
    w_s, b_s = sample if sample is not None else (None, None)
    n_s = 0 if w_s is None else w_s.shape[0]
    nbytes = encode_topk_workspace_bytes(B, H, D, k, n_s)
    ws = _workspace(x.device, nbytes)
    check(load().qsae_encode_topk(x.data_ptr(), w_bf16.data_ptr(), _ptr(w_f32), b_enc.data_ptr(), _ptr(w_s),
                                  _ptr(b_s), n_s, B, H, D, k, act, 1 if exact else 0, vals.data_ptr(),
                                  idx.data_ptr(), _ptr(flags), ws.data_ptr(), ws.numel(), _stream()))
    return vals, idx, flags


def bsae_forward(x: torch.Tensor, w_bf16: torch.Tensor, w_f32: torch.Tensor | None, b_enc: torch.Tensor, k: int,
                 packed: torch.Tensor, n_bits: int, qstep: float, dec_bias: torch.Tensor | None, exact: bool = False,
                 want_flags: bool = False, sample=None):
    """BinarySAE.forward on device buffers -> (vals [B,k], idx [B,k], flags | None, recon [B,D])."""
    _need_cuda(x, w_bf16, w_f32, b_enc, packed, dec_bias)
    B, D = x.shape
    H = w_bf16.shape[0]
    assert x.dtype == torch.float32 and w_bf16.dtype == torch.bfloat16 and b_enc.dtype == torch.float32
    vals = torch.empty((B, k), dtype=torch.float32, device=x.device)
    idx = torch.empty((B, k), dtype=torch.int32, device=x.device)
    recon = torch.empty((B, D), dtype=torch.float32, device=x.device)
    flags = torch.empty((B,), dtype=torch.int32, device=x.device) if want_flags else None
    if B == 0:
        return vals, idx, flags, recon
    w_s, b_s = sample if sample is not None else (None, None)
    n_s = 0 if w_s is None else w_s.shape[0]
    ws = _workspace(x.device, encode_topk_workspace_bytes(B, H, D, k, n_s))
    check(load().qsae_bsae_forward(x.data_ptr(), w_bf16.data_ptr(), _ptr(w_f32), b_enc.data_ptr(), _ptr(w_s), _ptr(b_s),
                                   n_s, B, H, D, k, 1 if exact else 0, packed.data_ptr(), n_bits, float(qstep),
                                   _ptr(dec_bias), vals.data_ptr(), idx.data_ptr(), _ptr(flags), recon.data_ptr(),
                                   ws.data_ptr(), ws.numel(), _stream()))
    return vals, idx, flags, recon


def encode_dense_tc(x: torch.Tensor, w_bf16: torch.Tensor, b_enc: torch.Tensor, act: int = ACT_NONE) -> torch.Tensor:
    """Diagnostic: dense z [B,H] straight from the tcgen05 encoder kernel."""
    _need_cuda(x, w_bf16, b_enc)
    B, D = x.shape
    H = w_bf16.shape[0]
    z = torch.empty((B, H), dtype=torch.float32, device=x.device)
    ws = _workspace(x.device, encode_topk_workspace_bytes(B, H, D, 1))
    check(load().qsae_encode_dense_tc(x.data_ptr(), w_bf16.data_ptr(), b_enc.data_ptr(), B, H, D, act,
                                      z.data_ptr(), ws.data_ptr(), ws.numel(), _stream()))
    return z


def encode_dense(x: torch.Tensor, w_f32: torch.Tensor, b_enc: torch.Tensor | None, act: int = ACT_NONE,
                 rows: torch.Tensor | None = None) -> torch.Tensor:
    _need_cuda(x, w_f32, b_enc, rows)
    R = x.shape[0] if rows is None else rows.numel()
    H, D = w_f32.shape
    z = torch.empty((R, H), dtype=torch.float32, device=x.device)
    check(load().qsae_encode_dense_f32(x.data_ptr(), _ptr(rows), R, w_f32.data_ptr(), _ptr(b_enc), H, D, act,
                                       z.data_ptr(), _stream()))
    return z


def topk_dense(z: torch.Tensor, k: int):
    _need_cuda(z)
    R, H = z.shape
    vals = torch.empty((R, k), dtype=torch.float32, device=z.device)
    idx = torch.empty((R, k), dtype=torch.int32, device=z.device)
    if R == 0:
        return vals, idx
    n = _sz(0)
    check(load().qsae_topk_dense_workspace_bytes(R, H, k, C.byref(n)))
    ws = _workspace(z.device, int(n.value))
    check(load().qsae_topk_dense(z.data_ptr(), R, H, k, vals.data_ptr(), idx.data_ptr(), ws.data_ptr(),
                                 ws.numel(), _stream()))
    return vals, idx


def _decode(fn_name: str, vals, idx, dict_t, H, D, scale, bias):
    _need_cuda(vals, idx, dict_t, bias)
    B, k = vals.shape
    recon = torch.empty((B, D), dtype=torch.float32, device=vals.device)
    check(getattr(load(), fn_name)(vals.data_ptr(), idx.data_ptr(), B, k, dict_t.data_ptr(), H, D, float(scale),
                                   _ptr(bias), recon.data_ptr(), _stream()))
    return recon


def decode_int4(vals, idx, packed, H, D, scale, bias):
    return _decode("qsae_decode_int4", vals, idx, packed, H, D, scale, bias)


def decode_int8(vals, idx, rows_i8, H, D, scale, bias):
    return _decode("qsae_decode_int8", vals, idx, rows_i8, H, D, scale, bias)


def decode_rows_f32(vals, idx, rows, H, D, scale, bias):
    return _decode("qsae_decode_rows_f32", vals, idx, rows, H, D, scale, bias)


def densify(vals: torch.Tensor, idx: torch.Tensor, H: int) -> torch.Tensor:
    _need_cuda(vals, idx)
    B, k = vals.shape
    dense = torch.empty((B, H), dtype=torch.float32, device=vals.device)
    check(load().qsae_densify(vals.data_ptr(), idx.data_ptr(), B, k, H, dense.data_ptr(), _stream()))
    return dense


def pack_matryoshka(weight: torch.Tensor, weight_mirror: torch.Tensor, level_start: torch.Tensor,
                    level_factor: torch.Tensor):
    """-> (packed [H, D/16] int32 (2-bit codes), scale [H] f32)"""
    _need_cuda(weight, weight_mirror, level_start, level_factor)
    H, D = weight.shape
    packed = torch.empty((H, D // 16), dtype=torch.int32, device=weight.device)
    scale = torch.empty((H,), dtype=torch.float32, device=weight.device)
    check(load().qsae_pack_matryoshka(weight.data_ptr(), weight_mirror.data_ptr(), H, D, level_start.data_ptr(),
                                      level_factor.data_ptr(), level_factor.numel(), packed.data_ptr(),
                                      scale.data_ptr(), _stream()))
    return packed, scale


def max_row_norm(w_f32: torch.Tensor) -> torch.Tensor:
    _need_cuda(w_f32)
    out = torch.zeros(1, dtype=torch.float32, device=w_f32.device)
    check(load().qsae_max_row_norm(w_f32.data_ptr(), w_f32.shape[0], w_f32.shape[1], out.data_ptr(), _stream()))
    return out


def decode_matryoshka_lists(lists, counts, cap, packed, scale, level_start, n_levels, H, D, dec_bias):
    _need_cuda(lists, counts, packed, scale, level_start, dec_bias)
    B = counts.shape[0]
    result = torch.empty((n_levels, B, D), dtype=torch.float32, device=lists.device)
    level_count = torch.zeros((n_levels,), dtype=torch.int64, device=lists.device)
    n = _sz(0)
    check(load().qsae_decode_matryoshka_lists_workspace_bytes(C.byref(n)))
    ws = _workspace(lists.device, int(n.value))
    check(load().qsae_decode_matryoshka_lists(lists.data_ptr(), counts.data_ptr(), cap, B, packed.data_ptr(),
                                              scale.data_ptr(), level_start.data_ptr(), n_levels, H, D, _ptr(dec_bias),
                                              result.data_ptr(), level_count.data_ptr(), ws.data_ptr(), ws.numel(),
                                              _stream()))
    return result, level_count


def matryoshka_forward(x, w_bf16, b_enc, packed, scale, level_start, n_levels, dec_bias, w_f32=None, w_norm_max=None,
                       active_cap: int = 0, want_residual: bool = False):
    """-> (result [n_levels, B, D] f32, level_count [n_levels] int64, overflow [1] int32)
    active_cap > 0: additionally (active_idx [B, active_cap] int32 with -1 in empty slots, active_cnt [B] int32).
    want_residual: additionally (x - result[-1]) * 2 [B, D], the next rq_sae stage's input, as the last element."""
    _need_cuda(x, w_bf16, b_enc, packed, scale, level_start, dec_bias)
    B, D = x.shape
    H = w_bf16.shape[0]
    result = torch.empty((n_levels, B, D), dtype=torch.float32, device=x.device)
    counts = torch.empty((n_levels,), dtype=torch.int64, device=x.device)
    overflow = torch.empty((1,), dtype=torch.int32, device=x.device)
    a_idx = torch.empty((B, active_cap), dtype=torch.int32, device=x.device) if active_cap > 0 else None
    a_cnt = torch.zeros((B,), dtype=torch.int32, device=x.device) if active_cap > 0 else None
    resid = torch.empty((B, D), dtype=torch.float32, device=x.device) if want_residual else None
    if B == 0:
        out = (result, counts.zero_(), overflow.zero_())
        out = out + (a_idx, a_cnt) if active_cap > 0 else out
        return out + (resid,) if want_residual else out
    n = _sz(0)
    check(load().qsae_matryoshka_workspace_bytes(B, H, D, C.byref(n)))
    ws = _workspace(x.device, int(n.value))
    check(load().qsae_matryoshka_forward_active(x.data_ptr(), w_bf16.data_ptr(), _ptr(w_f32), _ptr(w_norm_max),
                                                b_enc.data_ptr(), packed.data_ptr(), scale.data_ptr(),
                                                level_start.data_ptr(), n_levels, _ptr(dec_bias), B, H, D,
                                                result.data_ptr(), counts.data_ptr(), overflow.data_ptr(),
                                                _ptr(a_idx), active_cap, _ptr(a_cnt), _ptr(resid), ws.data_ptr(), ws.numel(),
                                                _stream()))
    out = (result, counts, overflow, a_idx, a_cnt) if active_cap > 0 else (result, counts, overflow)
    return out + (resid,) if want_residual else out


def activation_counts(idx: torch.Tensor, vals: torch.Tensor | None, counts: torch.Tensor) -> None:
    """counts [H] int64 += rows in which each latent is active (idx [B, cap] int32, -1 = empty; vals: active iff > 0)."""
    _need_cuda(idx, vals, counts)
    assert idx.dtype == torch.int32 and counts.dtype == torch.int64 and idx.dim() == 2
    B, cap = idx.shape
    check(load().qsae_activation_counts(idx.data_ptr(), _ptr(vals), B, cap, counts.numel(), counts.data_ptr(), _stream()))


def coactivation(idx: torch.Tensor, vals: torch.Tensor | None, cooc: torch.Tensor) -> None:
    """cooc [H, H] int32 += A^T A of the boolean activity described by the lists."""
    _need_cuda(idx, vals, cooc)
    assert idx.dtype == torch.int32 and cooc.dtype == torch.int32 and cooc.dim() == 2 and cooc.shape[0] == cooc.shape[1]
    B, cap = idx.shape
    check(load().qsae_coactivation(idx.data_ptr(), _ptr(vals), B, cap, cooc.shape[0], cooc.data_ptr(), _stream()))


def coactivation_dense(mask: torch.Tensor, cooc: torch.Tensor, counts: torch.Tensor | None = None) -> None:
    """cooc [H, H] int32 += mask^T mask and counts [H] int64 += mask.sum(0), for a bf16 0/1 activity mask [K, H]
    (tensor cores; K <= 2^24, H % 8 == 0)."""
    _need_cuda(mask, cooc, counts)
    assert mask.dtype == torch.bfloat16 and mask.dim() == 2 and cooc.dtype == torch.int32
    K, H = mask.shape
    assert cooc.shape == (H, H) and (counts is None or (counts.dtype == torch.int64 and counts.numel() == H))
    check(load().qsae_coactivation_dense(mask.data_ptr(), K, H, cooc.data_ptr(), _ptr(counts), _stream()))


def sq_error_accumulate(a: torch.Tensor, b: torch.Tensor, out: torch.Tensor) -> None:
    """out (device float64 scalar) += sum (a - b)^2."""
    _need_cuda(a, b, out)
    assert a.dtype == torch.float32 and b.dtype == torch.float32 and out.dtype == torch.float64 and a.numel() == b.numel()
    check(load().qsae_sq_error_accumulate(a.data_ptr(), b.data_ptr(), a.numel(), out.data_ptr(), _stream()))


# ---- training-side pieces adjacent to the forward (SURVEY 8f-4; csrc/train.cu) ----------------

def _f32c(*ts):
    for t in ts:
        if t is not None:
            assert t.dtype == torch.float32 and t.is_contiguous(), "float32 contiguous tensors expected"


def rows_scatter_add(coef, idx: torch.Tensor, src: torch.Tensor, dst: torch.Tensor, scale: float = 1.0, dst_col=None) -> None:
    """dst[idx[b,j], :] += scale * coef[b,j] * src[b, :] (coef None = 1); dst_col[idx[b,j]] += scale * coef[b,j]."""
    _need_cuda(coef, idx, src, dst, dst_col)
    _f32c(coef, src, dst, dst_col)
    assert idx.dtype == torch.int32 and idx.is_contiguous() and idx.dim() == 2 and src.dim() == 2 and dst.dim() == 2
    B, k = idx.shape
    assert src.shape[0] == B and src.shape[1] == dst.shape[1] and (coef is None or tuple(coef.shape) == (B, k))
    check(load().qsae_rows_scatter_add(_ptr(coef), idx.data_ptr(), src.data_ptr(), B, k, src.shape[1], dst.shape[0], float(scale),
                                       dst.data_ptr(), _ptr(dst_col), _stream()))


def rows_gather_dot(g: torch.Tensor, rows: torch.Tensor, idx: torch.Tensor, scale: float = 1.0) -> torch.Tensor:
    """out[b,j] = scale * <g[b,:], rows[idx[b,j], :]>."""
    _need_cuda(g, rows, idx)
    _f32c(g, rows)
    assert idx.dtype == torch.int32 and idx.is_contiguous() and idx.dim() == 2 and g.shape[1] == rows.shape[1]
    B, k = idx.shape
    out = torch.zeros((B, k), dtype=torch.float32, device=g.device)
    check(load().qsae_rows_gather_dot(g.data_ptr(), rows.data_ptr(), idx.data_ptr(), B, k, g.shape[1], rows.shape[0], float(scale),
                                      out.data_ptr(), _stream()))
    return out


def column_sum(src: torch.Tensor, scale: float = 1.0, out: torch.Tensor | None = None) -> torch.Tensor:
    """out[c] += scale * sum_r src[r, c] (out None: a fresh zero vector)."""
    _need_cuda(src, out)
    _f32c(src, out)
    R, Cn = src.shape
    if out is None:
        out = torch.zeros(Cn, dtype=torch.float32, device=src.device)
    check(load().qsae_column_sum(src.data_ptr(), R, Cn, float(scale), out.data_ptr(), _stream()))
    return out


def bsae_logit_grad(logits: torch.Tensor, G: torch.Tensor | None, D: int, n_bits: int, grad_polarize, grad: torch.Tensor,
                    accumulate: bool) -> None:
    """grad_logits (=|+=) (G c_i + gp 2^i (1 - 2p) / N) p (1 - p); grad_polarize: python float or 0-d device tensor."""
    _need_cuda(logits, G, grad)
    _f32c(logits, G, grad)
    H = logits.shape[0]
    assert logits.shape[1] == D * n_bits and grad.shape == logits.shape
    gp_dev, gp_host = None, 0.0
    if isinstance(grad_polarize, torch.Tensor):
        _need_cuda(grad_polarize)
        assert grad_polarize.dtype == torch.float32 and grad_polarize.numel() == 1
        gp_dev = grad_polarize
    else:
        gp_host = float(grad_polarize)
    check(load().qsae_bsae_logit_grad(logits.data_ptr(), _ptr(G), H, D, n_bits, _ptr(gp_dev), gp_host, int(accumulate),
                                      grad.data_ptr(), _stream()))


def _level_array(level_start_host):
    n = len(level_start_host) - 1
    return n, (C.c_int * (n + 1))(*[int(v) for v in level_start_host])


def matryoshka_backward_scatter(active_idx: torch.Tensor, grad_levels, level_start_host, M: torch.Tensor, z2: torch.Tensor) -> None:
    """M[h,:] += grad_levels[level(h)][b,:] for every active (b,h); z2[h] += 1."""
    _need_cuda(active_idx, M, z2, *grad_levels)
    _f32c(M, *grad_levels)
    assert active_idx.dtype == torch.int32 and active_idx.is_contiguous() and z2.dtype == torch.int32
    B, cap = active_idx.shape
    H, D = M.shape
    n, ls = _level_array(level_start_host)
    assert len(grad_levels) == n and all(tuple(g.shape) == (B, D) for g in grad_levels)
    ptrs = (_vp * n)(*[g.data_ptr() for g in grad_levels])
    check(load().qsae_matryoshka_backward_scatter(active_idx.data_ptr(), B, cap, H, D, ptrs, ls, n, M.data_ptr(), z2.data_ptr(),
                                                  _stream()))


def matryoshka_backward_finish(w, w_mirror, M, z2, alpha, level_start_host, c: float, joint_bits: int, grad_w, grad_w_mirror) -> None:
    """grad_w += (alpha M - sec Bsign(w)) s'(w), same for the mirror (M None: secant only; z2 None: STE only)."""
    _need_cuda(w, w_mirror, M, z2, alpha, grad_w, grad_w_mirror)
    _f32c(w, w_mirror, M, alpha, grad_w, grad_w_mirror)
    H, D = w.shape
    n, ls = _level_array(level_start_host)
    check(load().qsae_matryoshka_backward_finish(w.data_ptr(), w_mirror.data_ptr(), _ptr(M), _ptr(z2), alpha.data_ptr(), ls, n, H, D,
                                                 float(c), int(joint_bits), grad_w.data_ptr(), grad_w_mirror.data_ptr(), _stream()))


def matryoshka_backward_dense(mask: torch.Tensor, grad_levels, level_start_host, w, w_mirror, alpha, exact: bool, grad_w,
                              grad_w_mirror) -> torch.Tensor:
    """grad_w += alpha M s'(w), same for the mirror, M[h,:] = mask[:,h]^T grad_levels[level(h)], from a bf16 0/1 mask
    [B, H] (tensor cores; exact: three bf16 parts of each gradient). -> z2 [H] int32 = mask.sum(0)."""
    _need_cuda(mask, w, w_mirror, alpha, grad_w, grad_w_mirror, *grad_levels)
    _f32c(w, w_mirror, alpha, grad_w, grad_w_mirror, *grad_levels)
    assert mask.dtype == torch.bfloat16 and mask.dim() == 2
    B, H = mask.shape
    D = w.shape[1]
    n, ls = _level_array(level_start_host)
    assert len(grad_levels) == n and all(tuple(g.shape) == (B, D) for g in grad_levels)
    assert tuple(w.shape) == (H, D) and grad_w.shape == w.shape and w_mirror.shape == w.shape and grad_w_mirror.shape == w.shape
    nb = _sz(0)
    check(load().qsae_matryoshka_backward_dense_workspace_bytes(B, D, n, int(bool(exact)), C.byref(nb)))
    ws = _workspace(mask.device, int(nb.value))
    z2 = torch.empty((H,), dtype=torch.int32, device=mask.device)
    ptrs = (_vp * n)(*[g.data_ptr() for g in grad_levels])
    check(load().qsae_matryoshka_backward_dense(mask.data_ptr(), B, H, D, ptrs, ls, n, w.data_ptr(), w_mirror.data_ptr(),
                                                alpha.data_ptr(), int(bool(exact)), grad_w.data_ptr(), grad_w_mirror.data_ptr(),
                                                z2.data_ptr(), ws.data_ptr(), int(nb.value), _stream()))
    return z2


def _rigl_ws(device) -> torch.Tensor:
    n = _sz(0)
    check(load().qsae_rigl_workspace_bytes(C.byref(n)))
    return _workspace(device, int(n.value))


def rigl_init_mask(weight: torch.Tensor, mask: torch.Tensor, n_inactive: int) -> None:
    """In place: the n_inactive smallest |w| -> mask 0; weight *= mask (sae/ternary.py:27-39)."""
    _need_cuda(weight, mask)
    _f32c(weight, mask)
    D, H = weight.shape
    ws = _rigl_ws(weight.device)
    check(load().qsae_rigl_init_mask(weight.data_ptr(), mask.data_ptr(), D, H, int(n_inactive), ws.data_ptr(), ws.numel(), _stream()))


def rigl_update_mask(weight: torch.Tensor, mask: torch.Tensor, a_mean, d_mean, n_drop: int, n_grow: int) -> None:
    """In place RigL drop / grow step (sae/ternary.py:54-87)."""
    _need_cuda(weight, mask, a_mean, d_mean)
    _f32c(weight, mask, a_mean, d_mean)
    D, H = weight.shape
    assert a_mean is None or (a_mean.numel() == H and d_mean.numel() == D)
    ws = _rigl_ws(weight.device)
    check(load().qsae_rigl_update_mask(weight.data_ptr(), mask.data_ptr(), _ptr(a_mean), _ptr(d_mean), D, H, int(n_drop), int(n_grow),
                                       ws.data_ptr(), ws.numel(), _stream()))


def mul_inplace(a: torch.Tensor, b: torch.Tensor) -> None:
    _need_cuda(a, b)
    _f32c(a, b)
    assert a.numel() == b.numel()
    check(load().qsae_mul_inplace(a.data_ptr(), b.data_ptr(), a.numel(), _stream()))


def compact_dense(dense: torch.Tensor, mode: int, thr: float = 0.0, want_vals: bool = False, want_pairs: bool = False):
    """Dense [B, H] -> (idx [B, cap] int32 (-1 padded, ascending) | pairs [B, cap, 2], vals [B, cap] | None, cnt [B] int32).
    mode 0: entries != 0, mode 1: entries > thr. Two launches (count, then fill) with one host read of the largest
    count between them: the output shape depends on the data."""
    _need_cuda(dense)
    assert dense.dtype == torch.float32 and dense.is_contiguous() and dense.dim() == 2
    B, H = dense.shape
    cnt = torch.zeros((B,), dtype=torch.int32, device=dense.device)
    lib = load()
    check(lib.qsae_compact_dense(dense.data_ptr(), B, H, mode, float(thr), 0, None, None, None, cnt.data_ptr(), _stream()))
    cap = max(1, int(cnt.max().item())) if B else 1
    idx = None if want_pairs else torch.empty((B, cap), dtype=torch.int32, device=dense.device)
    pairs = torch.empty((B, cap, 2), dtype=torch.int32, device=dense.device) if want_pairs else None
    vals = torch.empty((B, cap), dtype=torch.float32, device=dense.device) if want_vals else None
    check(lib.qsae_compact_dense(dense.data_ptr(), B, H, mode, float(thr), cap, _ptr(idx), _ptr(vals), _ptr(pairs), cnt.data_ptr(),
                                 _stream()))
    return (pairs if want_pairs else idx), vals, cnt


def pack_ternary(w: torch.Tensor, threshold: float = 0.5, want_bf16: bool = True, want_rows: bool = False):
    """decoder.weight [D, H] -> (T bf16 [D, H] | None, T int8 rows [H, D] | None), T = sign(w) * (|w| >= thr)."""
    _need_cuda(w)
    D, H = w.shape
    assert w.dtype == torch.float32
    t_bf16 = torch.empty((D, H), dtype=torch.bfloat16, device=w.device) if want_bf16 else None
    t_rows = torch.empty((H, D), dtype=torch.int8, device=w.device) if want_rows else None
    check(load().qsae_pack_ternary(w.data_ptr(), D, H, float(threshold), _ptr(t_bf16), _ptr(t_rows), _stream()))
    return t_bf16, t_rows


def split_bf16(src: torch.Tensor, want_lo: bool = True):
    _need_cuda(src)
    assert src.dtype == torch.float32
    hi = torch.empty(src.shape, dtype=torch.bfloat16, device=src.device)
    lo = torch.empty(src.shape, dtype=torch.bfloat16, device=src.device) if want_lo else None
    check(load().qsae_split_bf16(src.data_ptr(), hi.data_ptr(), _ptr(lo), src.numel(), _stream()))
    return hi, lo


def decode_dense(a_hi: torch.Tensor, a_lo: torch.Tensor | None, b_t: torch.Tensor, bias: torch.Tensor | None = None):
    """out [B, N] = (a_hi (+ a_lo)) [B, K] @ b_t [N, K]^T (+ bias); bf16 operands, fp32 result."""
    _need_cuda(a_hi, a_lo, b_t, bias)
    B, K = a_hi.shape
    N = b_t.shape[0]
    assert a_hi.dtype == torch.bfloat16 and b_t.dtype == torch.bfloat16 and b_t.shape[1] == K
    out = torch.empty((B, N), dtype=torch.float32, device=a_hi.device)
    if B == 0:
        return out
    n = _sz(0)
    check(load().qsae_decode_dense_workspace_bytes(B, K, N, C.byref(n)))
    ws = _workspace(a_hi.device, int(n.value))
    check(load().qsae_decode_dense(a_hi.data_ptr(), _ptr(a_lo), b_t.data_ptr(), B, K, N, _ptr(bias), out.data_ptr(),
                                   ws.data_ptr(), ws.numel(), _stream()))
    return out


def split_bf16x3(src: torch.Tensor):
    """-> (hi, mid, lo) bf16 tensors with hi + mid + lo == src exactly."""
    _need_cuda(src)
    assert src.dtype == torch.float32
    parts = tuple(torch.empty(src.shape, dtype=torch.bfloat16, device=src.device) for _ in range(3))
    check(load().qsae_split_bf16x3(src.data_ptr(), parts[0].data_ptr(), parts[1].data_ptr(), parts[2].data_ptr(),
                                   src.numel(), _stream()))
    return parts


def tsae_forward(x: torch.Tensor, w_parts, b_enc: torch.Tensor, t_bf16: torch.Tensor, exact: bool):
    """w_parts: (bf16(W),) for the fast mode or split_bf16x3(W) for the exact mode.
    -> (h [B, H] f32 dense ReLU latents, recon [B, D] f32)"""
    w_hi = w_parts[0]
    w_mid, w_lo = (w_parts[1], w_parts[2]) if exact else (None, None)
    _need_cuda(x, w_hi, w_mid, w_lo, b_enc, t_bf16)
    B, D = x.shape
    H = t_bf16.shape[1]
    h = torch.empty((B, H), dtype=torch.float32, device=x.device)
    recon = torch.empty((B, D), dtype=torch.float32, device=x.device)
    if B == 0:
        return h, recon
    n = _sz(0)
    check(load().qsae_tsae_workspace_bytes(B, H, D, 1 if exact else 0, C.byref(n)))
    ws = _workspace(x.device, int(n.value))
    check(load().qsae_tsae_forward(x.data_ptr(), w_hi.data_ptr(), _ptr(w_mid), _ptr(w_lo), b_enc.data_ptr(),
                                   t_bf16.data_ptr(), B, H, D, 1 if exact else 0, h.data_ptr(), recon.data_ptr(),
                                   ws.data_ptr(), ws.numel(), _stream()))
    return h, recon


def pack_ternary_t(w: torch.Tensor, threshold: float = 0.5) -> torch.Tensor:
    """decoder.weight [D, H] -> T^T bf16 [H, D], T = sign(w) * (|w| >= thr) (B operand of the t_sae backward)."""
    _need_cuda(w)
    assert w.dtype == torch.float32
    D, H = w.shape
    t_t = torch.empty((H, D), dtype=torch.bfloat16, device=w.device)
    check(load().qsae_pack_ternary_t(w.data_ptr(), D, H, float(threshold), t_t.data_ptr(), _stream()))
    return t_t


def _bf16_parts(parts, what: str):
    parts = tuple(parts)
    if len(parts) not in (1, 3):
        raise ValueError(f"{what}: 1 or 3 bf16 parts expected, got {len(parts)}")
    _need_cuda(*parts)
    if any(p.dtype != torch.bfloat16 or p.dim() != 2 or p.shape != parts[0].shape for p in parts):
        raise ValueError(f"{what}: parts must be bf16 matrices of one shape")
    return parts


def wgrad(a_parts, b_parts, a_kmajor: bool = False) -> torch.Tensor:
    """c [M, N] fp32 = sum_k A(k, m) B(k, n) on the tensor cores (qsae_wgrad). b_parts: bf16 [K, N];
    a_parts: bf16 [K, M], or [M, K] with a_kmajor. One part each (one bf16 product) or three (split_bf16x3 parts:
    the six products above 2^-24 in one fp32 accumulator)."""
    a_parts = _bf16_parts(a_parts, "wgrad A")
    b_parts = _bf16_parts(b_parts, "wgrad B")
    if len(a_parts) != len(b_parts):
        raise ValueError("wgrad: A and B need the same number of parts")
    K, N = b_parts[0].shape
    M, Ka = (a_parts[0].shape if a_kmajor else a_parts[0].shape[::-1])
    if Ka != K:
        raise ValueError(f"wgrad: contraction lengths differ ({Ka} vs {K})")
    c = torch.empty((M, N), dtype=torch.float32, device=b_parts[0].device)
    n = len(a_parts)
    ap = (_vp * n)(*[p.data_ptr() for p in a_parts])
    bp = (_vp * n)(*[p.data_ptr() for p in b_parts])
    check(load().qsae_wgrad(ap, bp, n, M, N, K, 1 if a_kmajor else 0, c.data_ptr(), _stream()))
    return c


def tsae_backward(x: torch.Tensor, h: torch.Tensor, g_recon: torch.Tensor, g_h: torch.Tensor | None, t_t: torch.Tensor,
                  mask: torch.Tensor | None, w_parts, exact: bool, want_grad_x: bool):
    """Backward of t_sae's forward (qsae_tsae_backward). w_parts: (bf16(W_enc),) or split_bf16x3(W_enc), used for
    grad_x only. -> (grad W_enc [H, D], grad b_enc [H], grad W_dec [D, H], grad x [B, D] | None)"""
    _need_cuda(x, h, g_recon, g_h, t_t, mask)
    _f32c(x, h, g_recon, g_h, mask)
    B, D = x.shape
    H = h.shape[1]
    assert h.shape == (B, H) and g_recon.shape == (B, D) and t_t.shape == (H, D) and t_t.dtype == torch.bfloat16
    assert g_h is None or g_h.shape == (B, H)
    assert mask is None or mask.shape == (D, H)
    w = tuple(w_parts) if want_grad_x else (None, None, None)
    if want_grad_x:
        _need_cuda(*w)
        if len(w) != (3 if exact else 1):
            raise ValueError("tsae_backward: grad_x needs the encoder weight as 3 bf16 parts (exact) or 1 (fast)")
        w = w + (None,) * (3 - len(w))
    dev = x.device
    gwe = torch.empty((H, D), dtype=torch.float32, device=dev)
    gbe = torch.empty((H,), dtype=torch.float32, device=dev)
    gwd = torch.empty((D, H), dtype=torch.float32, device=dev)
    gx = torch.empty((B, D), dtype=torch.float32, device=dev) if want_grad_x else None
    n = _sz(0)
    check(load().qsae_tsae_backward_workspace_bytes(B, H, D, 1 if exact else 0, C.byref(n)))
    ws = _workspace(dev, int(n.value))
    check(load().qsae_tsae_backward(x.data_ptr(), h.data_ptr(), g_recon.data_ptr(), _ptr(g_h), t_t.data_ptr(), _ptr(mask),
                                    _ptr(w[0]), _ptr(w[1]), _ptr(w[2]), B, H, D, 1 if exact else 0, gwe.data_ptr(),
                                    gbe.data_ptr(), gwd.data_ptr(), _ptr(gx), ws.data_ptr(), ws.numel(), _stream()))
    return gwe, gbe, gwd, gx


def baseline_backward_workspace_bytes(B: int, H: int, D: int, k: int) -> int:
    n = _sz(0)
    check(load().qsae_baseline_backward_workspace_bytes(B, H, D, k, C.byref(n)))
    return int(n.value)


def baseline_backward(x: torch.Tensor, vals: torch.Tensor, idx: torch.Tensor, g_recon: torch.Tensor,
                      g_h: torch.Tensor | None, g_vals: torch.Tensor | None, w_enc: torch.Tensor | None,
                      dec_rows: torch.Tensor, want_grad_x: bool):
    """Backward of baseline_sae's forward (qsae_baseline_backward): g_h = d loss / d h dense [B, H] or g_vals over the
    kept values [B, k] (at most one). dec_rows: decoder.weight^T [H, D]. Bit-deterministic.
    -> (grad W_enc [H, D], grad b_enc [H], grad W_dec [D, H], grad b_dec [D], grad x [B, D] | None)"""
    _need_cuda(x, vals, idx, g_recon, g_h, g_vals, w_enc, dec_rows)
    _f32c(x, vals, g_recon, g_h, g_vals, w_enc, dec_rows)
    B, D = x.shape
    H = dec_rows.shape[0]
    k = idx.shape[1]
    assert vals.shape == (B, k) and idx.shape == (B, k) and idx.dtype == torch.int32 and g_recon.shape == (B, D)
    assert dec_rows.shape == (H, D) and (w_enc is None or w_enc.shape == (H, D))
    assert g_h is None or g_h.shape == (B, H)
    assert g_vals is None or g_vals.shape == (B, k)
    if want_grad_x and w_enc is None:
        raise ValueError("baseline_backward: grad_x needs the encoder weight")
    dev = x.device
    gwe = torch.empty((H, D), dtype=torch.float32, device=dev)
    gbe = torch.empty((H,), dtype=torch.float32, device=dev)
    gwd = torch.empty((D, H), dtype=torch.float32, device=dev)
    gbd = torch.empty((D,), dtype=torch.float32, device=dev)
    gx = torch.empty((B, D), dtype=torch.float32, device=dev) if want_grad_x else None
    ws = _workspace(dev, baseline_backward_workspace_bytes(B, H, D, k))
    check(load().qsae_baseline_backward(x.data_ptr(), vals.data_ptr(), idx.data_ptr(), g_recon.data_ptr(), _ptr(g_h),
                                        _ptr(g_vals), _ptr(w_enc) if want_grad_x else None, dec_rows.data_ptr(), B, H, D, k,
                                        gwe.data_ptr(), gbe.data_ptr(), gwd.data_ptr(), gbd.data_ptr(), _ptr(gx),
                                        ws.data_ptr(), ws.numel(), _stream()))
    return gwe, gbe, gwd, gbd, gx


def baseline_backward_range_workspace_bytes(B: int, H_shard: int, D: int, k: int) -> int:
    n = _sz(0)
    check(load().qsae_baseline_backward_range_workspace_bytes(B, H_shard, D, k, C.byref(n)))
    return int(n.value)


def baseline_backward_range(x: torch.Tensor, vals: torch.Tensor, idx: torch.Tensor, g_recon: torch.Tensor,
                            g_vals: torch.Tensor | None, rows_shard: torch.Tensor, idx_begin: int):
    """One shard's part of baseline_backward (qsae_baseline_backward_range): the shard owns the latents [idx_begin,
    idx_begin + H_shard) and holds rows_shard = its decoder.weight^T [H_shard, D]; idx holds global indices. The outputs
    are bit-equal to the matching slices of baseline_backward's for the same inputs.
    -> (grad W_enc [H_shard, D], grad b_enc [H_shard], grad W_dec [D, H_shard], grad b_dec [D])"""
    _need_cuda(x, vals, idx, g_recon, g_vals, rows_shard)
    _f32c(x, vals, g_recon, g_vals, rows_shard)
    B, D = x.shape
    H = rows_shard.shape[0]
    k = idx.shape[1]
    assert vals.shape == (B, k) and idx.shape == (B, k) and idx.dtype == torch.int32 and g_recon.shape == (B, D)
    assert rows_shard.shape == (H, D) and (g_vals is None or g_vals.shape == (B, k))
    dev = x.device
    gwe = torch.empty((H, D), dtype=torch.float32, device=dev)
    gbe = torch.empty((H,), dtype=torch.float32, device=dev)
    gwd = torch.empty((D, H), dtype=torch.float32, device=dev)
    gbd = torch.empty((D,), dtype=torch.float32, device=dev)
    ws = _workspace(dev, baseline_backward_range_workspace_bytes(B, H, D, k))
    check(load().qsae_baseline_backward_range(x.data_ptr(), vals.data_ptr(), idx.data_ptr(), g_recon.data_ptr(),
                                              _ptr(g_vals), rows_shard.data_ptr(), B, H, int(idx_begin), D, k,
                                              gwe.data_ptr(), gbe.data_ptr(), gwd.data_ptr(), gbd.data_ptr(),
                                              ws.data_ptr(), ws.numel(), _stream()))
    return gwe, gbe, gwd, gbd


def bsae_backward_workspace_bytes(B: int, H: int, D: int, k: int, n_bits: int) -> int:
    n = _sz(0)
    check(load().qsae_bsae_backward_workspace_bytes(B, H, D, k, n_bits, C.byref(n)))
    return int(n.value)


def bsae_backward(x: torch.Tensor, vals: torch.Tensor, idx: torch.Tensor, g_recon: torch.Tensor, soft_rows: torch.Tensor,
                  logits: torch.Tensor, q: float, grad_polarize, w_enc: torch.Tensor | None, n_bits: int, want_grad_x: bool):
    """Bit-deterministic backward of b_sae's soft forward (qsae_bsae_backward). soft_rows: the soft dictionary [H, D];
    grad_polarize: python float or 0-d device tensor (read on the device, no host synchronisation).
    -> (grad W_enc [H, D], grad b_enc [H], grad logits [H, D n_bits], grad b_dec [D], grad x [B, D] | None)"""
    _need_cuda(x, vals, idx, g_recon, soft_rows, logits, w_enc)
    _f32c(x, vals, g_recon, soft_rows, logits, w_enc)
    B, D = x.shape
    H = soft_rows.shape[0]
    k = idx.shape[1]
    assert vals.shape == (B, k) and idx.shape == (B, k) and idx.dtype == torch.int32 and g_recon.shape == (B, D)
    assert soft_rows.shape == (H, D) and logits.shape == (H, D * n_bits) and (w_enc is None or w_enc.shape == (H, D))
    if want_grad_x and w_enc is None:
        raise ValueError("bsae_backward: grad_x needs the encoder weight")
    gp_dev, gp_host = None, 0.0
    if isinstance(grad_polarize, torch.Tensor):
        _need_cuda(grad_polarize)
        assert grad_polarize.dtype == torch.float32 and grad_polarize.numel() == 1
        gp_dev = grad_polarize
    else:
        gp_host = float(grad_polarize)
    dev = x.device
    gwe = torch.empty((H, D), dtype=torch.float32, device=dev)
    gbe = torch.empty((H,), dtype=torch.float32, device=dev)
    glog = torch.empty((H, D * n_bits), dtype=torch.float32, device=dev)
    gbd = torch.empty((D,), dtype=torch.float32, device=dev)
    gx = torch.empty((B, D), dtype=torch.float32, device=dev) if want_grad_x else None
    ws = _workspace(dev, bsae_backward_workspace_bytes(B, H, D, k, n_bits))
    check(load().qsae_bsae_backward(x.data_ptr(), vals.data_ptr(), idx.data_ptr(), g_recon.data_ptr(), soft_rows.data_ptr(),
                                    logits.data_ptr(), float(q), _ptr(gp_dev), gp_host, _ptr(w_enc) if want_grad_x else None,
                                    B, H, D, k, n_bits, gwe.data_ptr(), gbe.data_ptr(), glog.data_ptr(), gbd.data_ptr(),
                                    _ptr(gx), ws.data_ptr(), ws.numel(), _stream()))
    return gwe, gbe, glog, gbd, gx


def pack_candidates(vals: torch.Tensor, idx: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    """(vals, idx) [B, k] -> [B, k, 2] int32 entries {float bits, index}: one all-gather operand
    (or, with `out`, written straight into this rank's peer-exchange buffer)."""
    _need_cuda(vals, idx, out)
    if out is None:
        out = torch.empty(tuple(vals.shape) + (2,), dtype=torch.int32, device=vals.device)
    assert out.dtype == torch.int32 and out.numel() == 2 * vals.numel()
    check(load().qsae_pack_candidates(vals.data_ptr(), idx.data_ptr(), vals.numel(), out.data_ptr(), _stream()))
    return out


def merge_candidates(cand_all: torch.Tensor, shard_latents: int, k_out: int, truncated: bool = False):
    """cand_all [G, B, k_in, 2] int32 (gathered pack_candidates outputs) -> global (vals, idx) [B, k_out].
    truncated=True (the shards sent fewer candidates than they hold): -> (vals, idx, incomplete [1] int32);
    incomplete != 0 means some shard's list was used up and the exchange must be repeated with full lists."""
    _need_cuda(cand_all)
    G, B, k_in, two = cand_all.shape
    assert two == 2 and cand_all.dtype == torch.int32
    vals = torch.empty((B, k_out), dtype=torch.float32, device=cand_all.device)
    idx = torch.empty((B, k_out), dtype=torch.int32, device=cand_all.device)
    flag = torch.zeros((1,), dtype=torch.int32, device=cand_all.device) if truncated else None
    if B == 0:
        return (vals, idx, flag) if truncated else (vals, idx)
    n = _sz(0)
    check(load().qsae_merge_candidates_workspace_bytes(B, C.byref(n)))
    ws = _workspace(cand_all.device, int(n.value))
    check(load().qsae_merge_candidates(cand_all.data_ptr(), G, B, k_in, shard_latents, k_out, vals.data_ptr(),
                                       idx.data_ptr(), _ptr(flag), ws.data_ptr(), ws.numel(), _stream()))
    return (vals, idx, flag) if truncated else (vals, idx)


def decode_range(vals, idx, dict_shard, shard_latents: int, idx_begin: int, D: int, scale: float, bias, n_bits: int,
                 out: torch.Tensor | None = None):
    """Partial reconstruction from the winners inside [idx_begin, idx_begin + shard_latents)."""
    _need_cuda(vals, idx, dict_shard, bias, out)
    B, k = vals.shape
    recon = torch.empty((B, D), dtype=torch.float32, device=vals.device) if out is None else out
    assert recon.dtype == torch.float32 and tuple(recon.shape) == (B, D)
    fn = load().qsae_decode_int4_range if n_bits <= 4 else load().qsae_decode_int8_range
    check(fn(vals.data_ptr(), idx.data_ptr(), B, k, dict_shard.data_ptr(), shard_latents, idx_begin, D, float(scale),
             _ptr(bias), recon.data_ptr(), _stream()))
    return recon


def decode_rows_f32_range(vals, idx, rows_shard, idx_begin: int, scale: float, bias, out: torch.Tensor | None = None):
    """Partial reconstruction from the winners inside [idx_begin, idx_begin + rows_shard.shape[0]) of an fp32 [H/G, D]
    row dictionary (the dictionary-sharded baseline_sae)."""
    _need_cuda(vals, idx, rows_shard, bias, out)
    B, k = vals.shape
    shard_latents, D = rows_shard.shape
    assert rows_shard.dtype == torch.float32
    recon = torch.empty((B, D), dtype=torch.float32, device=vals.device) if out is None else out
    assert recon.dtype == torch.float32 and tuple(recon.shape) == (B, D)
    check(load().qsae_decode_rows_f32_range(vals.data_ptr(), idx.data_ptr(), B, k, rows_shard.data_ptr(), shard_latents,
                                            idx_begin, D, float(scale), _ptr(bias), recon.data_ptr(), _stream()))
    return recon


def unpack_matryoshka_t(packed: torch.Tensor, D: int) -> torch.Tensor:
    """packed 2-bit codes [H, D/16] -> T^T bf16 [D, H] (entries -2, 0, +2)."""
    _need_cuda(packed)
    H = packed.shape[0]
    t = torch.empty((D, H), dtype=torch.bfloat16, device=packed.device)
    check(load().qsae_unpack_matryoshka_t(packed.data_ptr(), H, D, t.data_ptr(), _stream()))
    return t


def matryoshka_forward_dense(x, w_parts, b_enc, t_bf16, scale, level_start_dev, level_start_host, dec_bias,
                             mask=None, mask_col=0):
    """Dense q_sae forward -> (result [n_levels, B, D] f32, level_count [n_levels] int64).
    w_parts: (bf16(W),) or split_bf16x3(W) for fp32-accurate activity decisions. mask: bf16 [B, P] that also receives
    the activity (1.0 = active) in columns [mask_col, mask_col + H) (qsae_matryoshka_forward_dense_active)."""
    w_hi = w_parts[0]
    w_mid, w_lo = (w_parts[1], w_parts[2]) if len(w_parts) == 3 else (None, None)
    _need_cuda(x, w_hi, w_mid, w_lo, b_enc, t_bf16, scale, level_start_dev, dec_bias)
    B, D = x.shape
    H = t_bf16.shape[1]
    n_levels = len(level_start_host) - 1
    result = torch.empty((n_levels, B, D), dtype=torch.float32, device=x.device)
    counts = torch.zeros((n_levels,), dtype=torch.int64, device=x.device)
    if B == 0:
        return result, counts
    n = _sz(0)
    check(load().qsae_matryoshka_dense_workspace_bytes(B, H, D, C.byref(n)))
    ws = _workspace(x.device, int(n.value))
    starts = (_i * (n_levels + 1))(*[int(v) for v in level_start_host])
    if mask is not None:
        _need_cuda(mask)
        assert mask.dtype == torch.bfloat16 and mask.dim() == 2 and mask.shape[0] == B
        check(load().qsae_matryoshka_forward_dense_active(
            x.data_ptr(), w_hi.data_ptr(), _ptr(w_mid), _ptr(w_lo), b_enc.data_ptr(), t_bf16.data_ptr(), scale.data_ptr(),
            level_start_dev.data_ptr(), starts, n_levels, _ptr(dec_bias), B, H, D, result.data_ptr(), counts.data_ptr(),
            mask.data_ptr(), mask.shape[1], int(mask_col), ws.data_ptr(), ws.numel(), _stream()))
        return result, counts
    check(load().qsae_matryoshka_forward_dense(x.data_ptr(), w_hi.data_ptr(), _ptr(w_mid), _ptr(w_lo), b_enc.data_ptr(),
                                               t_bf16.data_ptr(),
                                               scale.data_ptr(), level_start_dev.data_ptr(), starts, n_levels,
                                               _ptr(dec_bias), B, H, D, result.data_ptr(), counts.data_ptr(),
                                               ws.data_ptr(), ws.numel(), _stream()))
    return result, counts


def residual_update(residual: torch.Tensor, recon: torch.Tensor) -> torch.Tensor:
    """(residual - recon) * 2 (sae/residual_quantized.py:67)."""
    _need_cuda(residual, recon)
    out = torch.empty_like(residual)
    check(load().qsae_residual_update(residual.data_ptr(), recon.data_ptr(), residual.numel(), out.data_ptr(), _stream()))
    return out


# ---- peer-memory exchange (dictionary-sharded forward without NCCL on the data path) --------------------------------
class _RawCudaBuffer:
    """A cudaMalloc'ed / IPC-mapped region exposed to torch through __cuda_array_interface__ (zero copy)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}


def peer_alloc(nbytes: int, device) -> tuple:
    """-> (ptr, uint8 tensor view, 64-byte IPC handle)"""
    ptr = _vp()
    with torch.cuda.device(device):       # cudaMalloc allocates on the current device
        check(load().qsae_peer_alloc(nbytes, C.byref(ptr)))
    handle = C.create_string_buffer(64)
    check(load().qsae_peer_export(ptr, handle))
    view = torch.as_tensor(_RawCudaBuffer(ptr.value, nbytes), device=device)
    return ptr.value, view, handle.raw


def peer_import(handle: bytes) -> int:
    ptr = _vp()
    check(load().qsae_peer_import(C.create_string_buffer(handle, 64), C.byref(ptr)))
    return ptr.value


def peer_close(ptr: int) -> None:
    check(load().qsae_peer_close(_vp(ptr)))


def peer_free(ptr: int) -> None:
    check(load().qsae_peer_free(_vp(ptr)))


def peer_signal(targets: torch.Tensor, value: int) -> None:
    """targets: device int64 [G] addresses of this rank's flag inside every rank's buffer."""
    check(load().qsae_peer_signal(targets.data_ptr(), targets.numel(), value & 0xFFFFFFFF, _stream()))


def peer_wait(flags_ptr: int, n: int, value: int, timed_out: torch.Tensor) -> None:
    check(load().qsae_peer_wait(_vp(flags_ptr), n, value & 0xFFFFFFFF, timed_out.data_ptr(), _stream()))


def merge_candidates_peer(list_bases: torch.Tensor, B: int, k_in: int, shard_latents: int, k_out: int,
                          truncated: bool = False):
    """list_bases: device int64 [G]; list s of row r at list_bases[s] + r * k_in 8-byte entries (peer memory)."""
    dev = list_bases.device
    vals = torch.empty((B, k_out), dtype=torch.float32, device=dev)
    idx = torch.empty((B, k_out), dtype=torch.int32, device=dev)
    flag = torch.zeros((1,), dtype=torch.int32, device=dev) if truncated else None
    if B == 0:
        return (vals, idx, flag) if truncated else (vals, idx)
    n = _sz(0)
    check(load().qsae_merge_candidates_workspace_bytes(B, C.byref(n)))
    ws = _workspace(dev, int(n.value))
    check(load().qsae_merge_candidates_peer(list_bases.data_ptr(), list_bases.numel(), B, k_in, shard_latents, k_out,
                                            vals.data_ptr(), idx.data_ptr(), _ptr(flag), ws.data_ptr(), ws.numel(), _stream()))
    return (vals, idx, flag) if truncated else (vals, idx)


def reduce_partials_peer(partial_bases: torch.Tensor, row_begin: int, rows: int, D: int) -> torch.Tensor:
    out = torch.empty((rows, D), dtype=torch.float32, device=partial_bases.device)
    check(load().qsae_reduce_partials_peer(partial_bases.data_ptr(), partial_bases.numel(), row_begin, rows, D,
                                           out.data_ptr(), _stream()))
    return out
