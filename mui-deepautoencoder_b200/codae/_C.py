"""ctypes binding of libcodae_b200.so (the C ABI declared in include/codae_b200.h).

PyTorch is only the plumbing here: it owns device memory and streams; every hot-path operation goes
through the C ABI with raw device pointers.  There is no CPU or eager-PyTorch fallback: importing
this module without the built library, or calling an op without a B200, raises.
"""
import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "libcodae_b200.so")

OK, EINVAL, EARCH, ECUDA, ENOMEM = 0, -1, -2, -3, -4
F32, BF16, F32X3 = 0, 1, 2     # F32X3: an fp32 tensor as three bf16 planes [3, ...] (hi, mid, lo)
ACT_NONE, ACT_RELU = 0, 1
METRIC_SQERR, METRIC_COSINE = 0, 1
VAR_REGRESSION, VAR_CLASSIFICATION = 0, 1
ENGINE_SIMT_F32, ENGINE_TCGEN05_BF16, ENGINE_TCGEN05_F32X3 = 0, 1, 2

_c = ctypes
_vp, _i, _i64, _u64, _f, _d, _sz = _c.c_void_p, _c.c_int, _c.c_int64, _c.c_uint64, _c.c_float, _c.c_double, _c.c_size_t

# name -> (restype, argtypes); must list every symbol of include/codae_b200.h (tests/test_abi.py checks)
SIGNATURES = {
    "codae_version": (_i, []),
    "codae_ctx_create": (_i, [_i, _c.POINTER(_vp)]),
    "codae_ctx_destroy": (_i, [_vp]),
    "codae_last_error": (_c.c_char_p, [_vp]),
    "codae_ctx_sm_count": (_i, [_vp]),
    "codae_ctx_set_option": (_i, [_vp, _i, _i]),
    "codae_ctx_get_option": (_i, [_vp, _i]),
    "codae_weights_written": (_i, [_vp, _vp]),
    "codae_linear_engine": (_i, [_vp, _i, _i, _i, _i]),
    "codae_mask_table_philox": (_i, [_vp, _u64, _i64, _i64, _i, _vp, _vp]),
    "codae_corrupt_fwd": (_i, [_vp, _vp, _i64, _i64, _vp, _i, _vp, _i, _i, _vp, _vp, _i, _vp, _i, _i64, _vp, _i64, _vp, _vp]),
    "codae_dense_masks": (_i, [_vp, _vp, _i, _vp, _i, _i, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "codae_mul_mask": (_i, [_vp, _vp, _vp, _vp, _i64, _vp]),
    "codae_loss_workspace_bytes": (_sz, [_vp]),
    "codae_mse_loss_fwd_bwd": (_i, [_vp, _vp, _i64, _vp, _vp, _i, _i64, _vp, _vp, _vp, _i, _i, _f, _vp, _i, _i64, _vp, _vp, _sz, _vp]),
    "codae_mixed_loss_fwd_bwd": (_i, [_vp, _vp, _vp, _i, _i, _i64, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "codae_mixed_monitor": (_i, [_vp, _vp, _vp, _i, _i, _i64, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "codae_linear_fwd": (_i, [_vp, _vp, _i64, _vp, _i64, _vp, _vp, _i64, _i, _i, _i, _i, _i, _i, _vp]),
    "codae_linear_dgrad": (_i, [_vp, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _i, _i, _i, _i, _i, _vp]),
    "codae_linear_wgrad": (_i, [_vp, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _i, _i, _i, _i, _vp]),
    "codae_linear_wgrad_sq_slots": (_i, [_vp, _i, _i, _i, _i]),
    "codae_linear_wgrad_sq": (_i, [_vp, _vp, _i64, _vp, _i64, _vp, _i64, _i, _i, _i, _i, _vp, _i, _vp]),
    "codae_linear_fwd_x3": (_i, [_vp, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _i64, _i, _i, _i, _i, _i, _vp]),
    "codae_linear_dgrad_x3": (_i, [_vp, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _vp, _i64, _i64, _i, _i, _i, _i, _vp]),
    "codae_linear_wgrad_x3": (_i, [_vp, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _i, _i, _i, _vp, _i, _vp]),
    "codae_split_x3": (_i, [_vp, _vp, _vp, _i64, _i64, _vp]),
    "codae_tiny_mlp_fwd": (_i, [_vp, _vp, _i, _vp, _vp, _i64, _i, _vp]),
    "codae_tiny_mlp_bwd": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _i64, _vp, _i64, _i, _vp]),
    "codae_cast_bf16": (_i, [_vp, _vp, _vp, _i64, _vp]),
    "codae_sqnorm_workspace_bytes": (_sz, [_vp]),
    "codae_grad_sqnorm": (_i, [_vp, _vp, _i64, _vp, _vp, _sz, _vp]),
    "codae_adam_step": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _d, _d, _d, _d, _d, _i, _d, _vp, _d, _vp, _vp]),
    "codae_clip_adam_step": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _d, _d, _d, _d, _d, _i, _d, _vp, _vp, _sz, _d, _vp, _vp]),
    "codae_adam_step_partials": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _d, _d, _d, _d, _d, _i, _d, _vp, _i, _vp, _d, _vp, _vp]),
    "codae_counter_add": (_i, [_vp, _vp, _i, _vp]),
    "codae_dp_workspace_bytes": (_sz, [_vp]),
    "codae_dp_shard_elems": (_i64, [_i64, _i]),
    "codae_dp_adam_step": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i64, _d, _d, _d, _d, _d, _i, _d, _vp, _vp, _sz, _d, _vp, _vp]),
    "codae_score_topk_workspace_bytes": (_sz, [_vp, _i, _i]),
    "codae_score_topk": (_i, [_vp, _vp, _i, _i64, _i64, _i, _i64, _vp, _i, _f, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "codae_score_topk_batched_workspace_bytes": (_sz, [_vp, _i, _i64, _i, _i, _i]),
    "codae_score_topk_batched": (_i, [_vp, _vp, _i, _i64, _i64, _i, _i64, _vp, _i, _f, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz,
                                      _vp]),
    "codae_score_topk_filtered": (_i, [_vp, _vp, _i, _i64, _i64, _i, _i64, _vp, _i, _f, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _sz,
                                       _vp]),
    "codae_score_topk_batched_filtered": (_i, [_vp, _vp, _i, _i64, _i64, _i, _i64, _vp, _i, _f, _i, _i, _vp, _vp, _i, _vp, _vp,
                                               _vp, _vp, _vp, _sz, _vp]),
    "codae_topk_merge": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "codae_score_rank": (_i, [_vp, _vp, _i, _i64, _i64, _i, _vp, _i, _f, _i, _vp, _vp, _i64, _vp, _vp]),
    "codae_row_sqnorm": (_i, [_vp, _vp, _i64, _i64, _i, _vp, _vp]),
    "codae_rank_count": (_i, [_vp, _vp, _i64, _i, _i64, _vp, _vp, _vp, _vp]),
    "codae_swap_build": (_i, [_vp, _vp, _vp, _i, _i64, _i64, _i, _i, _i, _i, _f, _vp, _i, _i64, _vp]),
    "codae_swap_error_topk": (_i, [_vp, _vp, _vp, _i, _i64, _i64, _i, _i, _i, _i, _f, _vp, _i64, _i64, _i, _vp, _vp, _vp,
                                   _sz, _vp]),
    "codae_swap_error_topk_filtered": (_i, [_vp, _vp, _vp, _i, _i64, _i64, _i, _i, _i, _i, _f, _vp, _i64, _i64, _i, _vp, _vp, _i,
                                            _vp, _vp, _vp, _sz, _vp]),
    "codae_swap_build_pairs": (_i, [_vp, _vp, _i64, _i, _vp, _i, _i64, _i64, _i64, _vp, _i, _vp, _i, _i, _i, _i, _f, _vp, _i, _i64,
                                    _vp]),
    "codae_swap_error_pairs": (_i, [_vp, _vp, _i64, _i, _vp, _i, _i64, _i64, _i64, _vp, _i, _vp, _i, _i, _i, _i, _f, _vp, _i64, _vp,
                                    _vp]),
    "codae_swap_pairs_topk": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
}

DP_MAX_WORLD = 8
DP_SIGNAL_BYTES = 512


class DpPeers(ctypes.Structure):
    """struct codae_dp_peers (include/codae_b200.h): every rank's gradient buffer, weight buffer and signal pad as device
    pointers valid in this process."""
    _fields_ = [("world", _c.c_int32), ("rank", _c.c_int32), ("grads", _vp * DP_MAX_WORLD), ("w_out", _vp * DP_MAX_WORLD),
                ("signals", _vp * DP_MAX_WORLD), ("grads_mc", _vp), ("w_mc", _vp)]


class TinyLayer(ctypes.Structure):
    """struct codae_tiny_layer (include/codae_b200.h)."""
    _fields_ = [("w_off", _i64), ("ld", _c.c_int32), ("bcol", _c.c_int32), ("in_", _c.c_int32), ("out", _c.c_int32),
                ("relu", _c.c_int32)]


TINY_MAX_LAYERS = 8
MIXED_MAX_VARIABLES = 64      # csrc/loss.cu: kMaxVar (variables per row, categories per classification variable)
MIXED_MAX_CATEGORIES = 64

_lib = None
_lock = threading.RLock()   # re-entrant: ctx() loads the library under the same lock
_ctxs = {}


def lib():
    """The loaded shared library.  Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        "libcodae_b200.so is not built (%s). Run `python __graft_entry__.py` or "
                        "`make -C mui-deepautoencoder_b200/csrc`. There is no CPU fallback." % LIB_PATH)
                l = ctypes.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(l, name)
                    fn.restype = res
                    fn.argtypes = args
                _lib = l
    return _lib


def ctx(device=None):
    """codae_ctx* for a CUDA device (one per process and device)."""
    if not torch.cuda.is_available():
        raise RuntimeError("codae: no CUDA device; the B200 path has no CPU fallback")
    dev = torch.cuda.current_device() if device is None else torch.device(device).index
    if dev is None:
        dev = torch.cuda.current_device()
    c = _ctxs.get(dev)
    if c is None:
        with _lock:
            c = _ctxs.get(dev)
            if c is None:
                out = _vp()
                rc = lib().codae_ctx_create(dev, ctypes.byref(out))
                if rc != OK:
                    raise RuntimeError("codae_ctx_create failed (%d): %s" % (rc, (lib().codae_last_error(None) or b"").decode()))
                c = out
                _ctxs[dev] = c
    return c


OPT_SPLITK, OPT_PDL, OPT_PERSISTENT, OPT_WEIGHT_PREFETCH, OPT_TMA_STORE, OPT_TMA_STORE_PERSISTENT, OPT_CTA_PAIR = 0, 1, 2, 3, 4, 5, 6


def set_option(device, option, value):
    """Tuning switches of the library (include/codae_b200.h: enum codae_option)."""
    c = ctx(device)
    check(lib().codae_ctx_set_option(c, option, 1 if value else 0), c)


def weights_written(device):
    """The current stream now waits for a weight writer on another stream: its next launch gets a full dependency."""
    c = ctx(device)
    check(lib().codae_weights_written(c, stream()), c)


def get_option(device, option):
    v = lib().codae_ctx_get_option(ctx(device), option)
    if v < 0:
        raise RuntimeError("codae: unknown option %d" % option)
    return v


def set_splitk(device, enabled):
    set_option(device, OPT_SPLITK, enabled)


def check(rc, c):
    if rc != OK:
        raise RuntimeError("libcodae_b200 error %d: %s" % (rc, (lib().codae_last_error(c) or b"").decode()))


def p(t):
    """Raw device pointer of a tensor (or NULL)."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def is_x3(t):
    """A CODAE_F32X3 matrix: three bf16 planes stacked along a leading dimension, [3, rows, pitch] (2-D bf16 tensors are plain
    bf16 matrices; the flat weight shadow [3, n] only ever goes to the optimizer wrappers)."""
    return t is not None and t.dtype == torch.bfloat16 and t.dim() == 3 and t.shape[0] == 3


def new_x3(shape, device):
    return torch.zeros((3,) + tuple(shape), dtype=torch.bfloat16, device=device)


def x3_to_f32(t):
    """fp32 value of a CODAE_F32X3 tensor (hi + mid + lo, exact in fp32)."""
    return (t[0].float() + t[1].float()) + t[2].float()


def dt(t):
    if is_x3(t):
        return F32X3
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise TypeError("codae: unsupported dtype %s" % t.dtype)


def ld(t):
    """Row pitch in elements (of one plane for CODAE_F32X3)."""
    return t.stride(1) if is_x3(t) else t.stride(0)


def _own_planes(t, B):
    """CODAE_F32X3 outputs of the elementwise kernels are [3, B, ld] with plane stride B * ld."""
    if is_x3(t) and t.stride(0) != B * t.stride(1):
        raise RuntimeError("codae: a CODAE_F32X3 output of this kernel must be a whole [3, B, ld] buffer (plane stride B * ld)")


def _dev_check(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("codae: tensor is not on a CUDA device; the B200 path has no CPU fallback")


# ---- thin typed wrappers (tensor in, kernel launch on the current stream) ---------------------------

def mask_table_philox(seed, first_obs, n_obs, nb_run, device):
    out = torch.empty((n_obs, nb_run), dtype=torch.int16, device=device)
    c = ctx(device)
    check(lib().codae_mask_table_philox(c, seed & 0xFFFFFFFFFFFFFFFF, first_obs, n_obs, nb_run, p(out), stream()), c)
    return out


def corrupt_fwd(data, batch_idx, B, mask_table, run, mask_bits, col_var, io, out_cx, out_x=None, out_mask_id=None):
    _dev_check(data, batch_idx, mask_table, out_cx)
    _own_planes(out_cx, B)
    c = ctx(data.device)
    check(lib().codae_corrupt_fwd(c, p(data), data.shape[0], data.stride(0), p(batch_idx), B, p(mask_table), mask_table.shape[1], run,
                                  p(mask_bits), p(col_var), io, p(out_cx), dt(out_cx), ld(out_cx), p(out_x),
                                  0 if out_x is None else out_x.stride(0), p(out_mask_id), stream()), c)


def dense_masks(batch_idx, B, mask_table, run, mask_bits, nb_missing, col_var, io, k_max, out_masks, out_fmask):
    _dev_check(mask_table, out_masks)
    c = ctx(mask_table.device)
    check(lib().codae_dense_masks(c, p(batch_idx), B, p(mask_table), mask_table.shape[1], run, p(mask_bits), p(nb_missing),
                                  p(col_var), io, k_max, p(out_masks), p(out_fmask), stream()), c)


def mul_mask(x, mask, out):
    _dev_check(x, mask, out)
    c = ctx(x.device)
    check(lib().codae_mul_mask(c, p(x), p(mask), p(out), x.numel(), stream()), c)


def loss_workspace(device):
    c = ctx(device)
    return torch.zeros(int(lib().codae_loss_workspace_bytes(c)), dtype=torch.uint8, device=device)


def mse_loss_fwd_bwd(x, batch_idx, y, mask_id, mask_bits, col_var, B, io, grad_scale, dy, acc, ws):
    _dev_check(x, y, acc, ws)
    if dy is not None:
        _own_planes(dy, B)
    c = ctx(x.device)
    check(lib().codae_mse_loss_fwd_bwd(c, p(x), x.stride(0), p(batch_idx), p(y), dt(y), y.stride(0), p(mask_id), p(mask_bits),
                                       p(col_var), B, io, grad_scale, p(dy), F32 if dy is None else dt(dy),
                                       0 if dy is None else ld(dy), p(acc), p(ws), ws.numel(), stream()), c)


def mixed_loss_fwd_bwd(x, y, var_pos, var_size, var_type, weight, dy, loss_out):
    _dev_check(x, y, dy)
    c = ctx(x.device)
    assert x.stride(0) == y.stride(0) == dy.stride(0)
    check(lib().codae_mixed_loss_fwd_bwd(c, p(x), p(y), x.shape[0], x.shape[1], x.stride(0), var_pos.numel(), p(var_pos),
                                         p(var_size), p(var_type), p(weight), p(dy), p(loss_out), stream()), c)


def mixed_monitor(x, y, var_pos, var_size, var_type, norm_scale, norm_min, norm_first, mask_id, mask_bits, nb_missing,
                  k_max, out_loss, acc):
    _dev_check(x, y, out_loss, acc)
    c = ctx(x.device)
    assert x.stride(0) == y.stride(0)
    check(lib().codae_mixed_monitor(c, p(x), p(y), x.shape[0], x.shape[1], x.stride(0), var_pos.numel(), p(var_pos),
                                    p(var_size), p(var_type), p(norm_scale), p(norm_min), norm_first, p(mask_id),
                                    p(mask_bits), p(nb_missing), k_max, p(out_loss), p(acc), stream()), c)


def linear_fwd(X, W, bias, Y, M, N, K, act, dtype):
    c = ctx(X.device)
    if dtype == F32X3:
        assert is_x3(X) and is_x3(W) and bias is None, "codae: the fp32-parity engine contracts CODAE_F32X3 operands (bias = augmented column)"
        check(lib().codae_linear_fwd_x3(c, p(X), ld(X), X.stride(0), p(W), ld(W), W.stride(0), p(Y), ld(Y),
                                        Y.stride(0) if is_x3(Y) else 0, M, N, K, act, dt(Y), stream()), c)
        return
    check(lib().codae_linear_fwd(c, p(X), X.stride(0), p(W), W.stride(0), p(bias), p(Y), Y.stride(0), M, N, K, act, dtype,
                                 dt(Y), stream()), c)


def linear_dgrad(dY, W, A_prev, dX, M, N, K, dtype):
    c = ctx(dY.device)
    if dtype == F32X3:
        assert is_x3(dY) and is_x3(W)
        hi = None if A_prev is None else (A_prev[0] if is_x3(A_prev) else A_prev)      # x > 0 <=> its hi plane > 0
        assert hi is None or hi.dtype == torch.bfloat16
        check(lib().codae_linear_dgrad_x3(c, p(dY), ld(dY), dY.stride(0), p(W), ld(W), W.stride(0), p(hi),
                                          0 if hi is None else hi.stride(0), p(dX), ld(dX), dX.stride(0) if is_x3(dX) else 0,
                                          M, N, K, dt(dX), stream()), c)
        return
    check(lib().codae_linear_dgrad(c, p(dY), dY.stride(0), p(W), W.stride(0), p(A_prev),
                                   0 if A_prev is None else A_prev.stride(0), p(dX), dX.stride(0), M, N, K, dtype, dt(dX),
                                   stream()), c)


def linear_wgrad(dY, X, dW, db, M, N, K, dtype):
    c = ctx(dY.device)
    if dtype == F32X3:
        assert is_x3(dY) and is_x3(X) and db is None, "codae: the fp32-parity engine takes the bias gradient from the augmented column"
        check(lib().codae_linear_wgrad_x3(c, p(dY), ld(dY), dY.stride(0), p(X), ld(X), X.stride(0), p(dW), dW.stride(0), M, N, K,
                                          None, 0, stream()), c)
        return
    check(lib().codae_linear_wgrad(c, p(dY), dY.stride(0), p(X), X.stride(0), p(dW), dW.stride(0), p(db), M, N, K, dtype,
                                   stream()), c)


def linear_wgrad_sq_slots(device, M, N, K, dtype):
    return int(lib().codae_linear_wgrad_sq_slots(ctx(device), M, N, K, dtype))


def linear_wgrad_sq(dY, X, dW, M, N, K, dtype, sq_partials):
    c = ctx(dY.device)
    if dtype == F32X3:
        assert is_x3(dY) and is_x3(X)
        check(lib().codae_linear_wgrad_x3(c, p(dY), ld(dY), dY.stride(0), p(X), ld(X), X.stride(0), p(dW), dW.stride(0), M, N, K,
                                          p(sq_partials), sq_partials.numel(), stream()), c)
        return
    check(lib().codae_linear_wgrad_sq(c, p(dY), dY.stride(0), p(X), X.stride(0), p(dW), dW.stride(0), M, N, K, dtype,
                                      p(sq_partials), sq_partials.numel(), stream()), c)


def split_x3(src, dst):
    """fp32 (contiguous, numel % 4 == 0) -> CODAE_F32X3 planes dst [3, ...] of the same per-plane shape."""
    assert dst.dtype == torch.bfloat16 and dst.shape[0] == 3 and src.dtype == torch.float32
    assert src.is_contiguous() and dst[0].is_contiguous() and dst[0].numel() == src.numel()
    c = ctx(src.device)
    check(lib().codae_split_x3(c, p(src), p(dst), src.numel(), dst.stride(0), stream()), c)


def dp_shard_elems(n, world):
    """Elements of the flat buffers every rank owns under the sharded data-parallel update (host arithmetic, no GPU needed)."""
    return int(lib().codae_dp_shard_elems(n, world))


def dp_workspace(device):
    c = ctx(device)
    return torch.zeros(int(lib().codae_dp_workspace_bytes(c)), dtype=torch.uint8, device=device)


def dp_peers(world, rank, grad_ptrs, w_ptrs, signal_ptrs, grads_mc=0, w_mc=0):
    """grads_mc / w_mc: NVSwitch multicast addresses of the gradient / weight buffers (0: peer loads and stores)."""
    pe = DpPeers()
    pe.world, pe.rank = world, rank
    pe.grads_mc, pe.w_mc = (int(grads_mc) or None), (int(w_mc) or None)
    for q in range(world):
        pe.grads[q], pe.w_out[q], pe.signals[q] = int(grad_ptrs[q]), int(w_ptrs[q]), int(signal_ptrs[q])
    return pe


def dp_adam_step(peers, pf, m, v, w_dtype, lr, beta1, beta2, eps, wd, step, max_norm, sqnorm_out, ws, grad_scale, step_dev=None):
    """Reduce-scatter + clip + Adam on this rank's shard + all-gather of the new weights, one kernel over peer memory."""
    _dev_check(pf, m, v, sqnorm_out, ws)
    c = ctx(pf.device)
    check(lib().codae_dp_adam_step(c, ctypes.byref(peers), p(pf), p(m), p(v), w_dtype, pf.numel(), lr, beta1, beta2, eps, wd, step,
                                   max_norm, p(sqnorm_out), p(ws), ws.numel(), grad_scale, p(step_dev), stream()), c)


def _ptr_array(tensors):
    return ctypes.cast((_vp * len(tensors))(*[t.data_ptr() for t in tensors]), _vp)


def tiny_mlp_fwd(layers, flat, acts, B):
    """layers: list of TinyLayer; acts: L+1 fp32 activation buffers with ONE common pitch (constant-1 columns set)."""
    c = ctx(flat.device)
    assert len({a.stride(0) for a in acts}) == 1 and all(a.dtype == torch.float32 for a in acts)
    arr = (TinyLayer * len(layers))(*layers)
    check(lib().codae_tiny_mlp_fwd(c, ctypes.cast(arr, _vp), len(layers), p(flat), _ptr_array(acts), acts[0].stride(0), B, stream()), c)


def tiny_mlp_bwd(layers, flat, gflat, acts, g3, B):
    """g3: the three rotating fp32 gradient buffers (dL/d(out_l) in g3[l % 3]; g3[(L-1) % 3] holds dL/dy)."""
    c = ctx(flat.device)
    assert len({a.stride(0) for a in acts}) == 1 and len({g.stride(0) for g in g3}) == 1 and len(g3) == 3
    arr = (TinyLayer * len(layers))(*layers)
    check(lib().codae_tiny_mlp_bwd(c, ctypes.cast(arr, _vp), len(layers), p(flat), p(gflat), _ptr_array(acts), acts[0].stride(0),
                                   _ptr_array(g3), g3[0].stride(0), B, stream()), c)


def cast_bf16(src, dst):
    c = ctx(src.device)
    check(lib().codae_cast_bf16(c, p(src), p(dst), src.numel(), stream()), c)


def sqnorm_workspace(device):
    c = ctx(device)
    return torch.zeros(int(lib().codae_sqnorm_workspace_bytes(c)), dtype=torch.uint8, device=device)


def grad_sqnorm(g, out, ws):
    c = ctx(g.device)
    check(lib().codae_grad_sqnorm(c, p(g), g.numel(), p(out), p(ws), ws.numel(), stream()), c)


def _shadow_dt(shadow, pf):
    """Weight copy the GEMMs read: None, bf16 [n], or CODAE_F32X3 planes [3, n] (contiguous)."""
    if shadow is None:
        return BF16
    if shadow.dim() == 2:
        assert shadow.dtype == torch.bfloat16 and shadow.shape == (3, pf.numel()) and shadow.is_contiguous()
        return F32X3
    assert shadow.dtype == torch.bfloat16 and shadow.numel() == pf.numel()
    return BF16


def adam_step(pf, g, m, v, shadow, lr, beta1, beta2, eps, wd, step, max_norm, sqnorm, grad_scale, step_dev=None):
    c = ctx(pf.device)
    check(lib().codae_adam_step(c, p(pf), p(g), p(m), p(v), p(shadow), _shadow_dt(shadow, pf), pf.numel(), lr, beta1, beta2, eps, wd, step, max_norm,
                                p(sqnorm), grad_scale, p(step_dev), stream()), c)


def clip_adam_step(pf, g, m, v, shadow, lr, beta1, beta2, eps, wd, step, max_norm, sqnorm_out, ws, grad_scale, step_dev=None):
    c = ctx(pf.device)
    check(lib().codae_clip_adam_step(c, p(pf), p(g), p(m), p(v), p(shadow), _shadow_dt(shadow, pf), pf.numel(), lr, beta1, beta2, eps, wd, step, max_norm,
                                     p(sqnorm_out), p(ws), ws.numel(), grad_scale, p(step_dev), stream()), c)


def adam_step_partials(pf, g, m, v, shadow, lr, beta1, beta2, eps, wd, step, max_norm, sq_partials, sqnorm_out, grad_scale,
                       step_dev=None):
    c = ctx(pf.device)
    check(lib().codae_adam_step_partials(c, p(pf), p(g), p(m), p(v), p(shadow), _shadow_dt(shadow, pf), pf.numel(), lr, beta1, beta2, eps, wd, step,
                                         max_norm, p(sq_partials), sq_partials.numel(), p(sqnorm_out), grad_scale,
                                         p(step_dev), stream()), c)


def counter_add(counter, delta):
    c = ctx(counter.device)
    check(lib().codae_counter_add(c, p(counter), delta, stream()), c)


def score_topk_workspace(device, Q, k):
    c = ctx(device)
    return torch.empty(int(lib().codae_score_topk_workspace_bytes(c, Q, k)), dtype=torch.uint8, device=device)


TOPK_MAX_EXCLUDE = 256       # include/codae_b200.h: CODAE_TOPK_MAX_EXCLUDE


def _n_exclude(exclude):
    """Columns of an exclusion tensor ([Q, m] or [m]); m == 0 is passed as no list (NULL, 0)."""
    m = 0 if exclude is None else int(exclude.shape[-1])
    return (exclude if m else None), m


def score_topk(catalog, E, row_offset, query, inv_scale, metric, k, out_score, out_idx, ws, allow=None, exclude=None):
    """allow: uint8 [n_rows] or None; exclude: int64 [Q, m] global indices (-1 padding) or None.  Without either, the
    unfiltered entry point (codae_score_topk)."""
    _dev_check(catalog, query, out_score, out_idx, ws, allow, exclude)
    c = ctx(catalog.device)
    if allow is None and exclude is None:
        check(lib().codae_score_topk(c, p(catalog), dt(catalog), catalog.shape[0], catalog.stride(0), E, row_offset, p(query),
                                     query.shape[0], inv_scale, metric, k, p(out_score), p(out_idx), p(ws), ws.numel(),
                                     stream()), c)
        return
    ex, m = _n_exclude(exclude)
    check(lib().codae_score_topk_filtered(c, p(catalog), dt(catalog), catalog.shape[0], catalog.stride(0), E, row_offset, p(query),
                                          query.shape[0], inv_scale, metric, k, p(allow), p(ex), m, p(out_score), p(out_idx),
                                          p(ws), ws.numel(), stream()), c)


TOPK_BATCHED_MAX_K = 64      # include/codae_b200.h: CODAE_TOPK_BATCHED_MAX_K


def score_topk_batched_workspace(catalog, E, Q, k):
    c = ctx(catalog.device)
    n = int(lib().codae_score_topk_batched_workspace_bytes(c, dt(catalog), catalog.shape[0], E, Q, k))
    return torch.empty(n, dtype=torch.uint8, device=catalog.device)


def score_topk_batched(catalog, E, row_offset, query, inv_scale, metric, k, out_score, out_idx, n_uncertified, uncertified, ws,
                       allow=None, exclude=None):
    """Tensor-core proposals + certification (codae_score_topk_batched).  n_uncertified: int32 [1], uncertified: int32 [Q].
    allow / exclude as in score_topk (codae_score_topk_batched_filtered when either is given)."""
    _dev_check(catalog, query, out_score, out_idx, n_uncertified, uncertified, ws, allow, exclude)
    assert n_uncertified.dtype == torch.int32 and uncertified.dtype == torch.int32 and uncertified.numel() >= query.shape[0]
    c = ctx(catalog.device)
    if allow is None and exclude is None:
        check(lib().codae_score_topk_batched(c, p(catalog), dt(catalog), catalog.shape[0], catalog.stride(0), E, row_offset,
                                             p(query), query.shape[0], inv_scale, metric, k, p(out_score), p(out_idx),
                                             p(n_uncertified), p(uncertified), p(ws), ws.numel(), stream()), c)
        return
    ex, m = _n_exclude(exclude)
    check(lib().codae_score_topk_batched_filtered(c, p(catalog), dt(catalog), catalog.shape[0], catalog.stride(0), E, row_offset,
                                                  p(query), query.shape[0], inv_scale, metric, k, p(allow), p(ex), m,
                                                  p(out_score), p(out_idx), p(n_uncertified), p(uncertified), p(ws), ws.numel(),
                                                  stream()), c)


def topk_merge(scores, idx, metric, out_score, out_idx):
    c = ctx(scores.device)
    G, Q, k = scores.shape
    check(lib().codae_topk_merge(c, p(scores), p(idx), G, Q, k, metric, p(out_score), p(out_idx), stream()), c)


def score_rank(catalog, E, query, inv_scale, metric, true_idx, subset_idx, out_rank):
    _dev_check(catalog, query, true_idx, out_rank)
    c = ctx(catalog.device)
    check(lib().codae_score_rank(c, p(catalog), dt(catalog), catalog.shape[0], catalog.stride(0), E, p(query),
                                 query.shape[0], inv_scale, metric, p(true_idx), p(subset_idx),
                                 0 if subset_idx is None else subset_idx.numel(), p(out_rank), stream()), c)


def row_sqnorm(X, E, out):
    """out[r] = sum_d X[r, d]^2 (f32 rows of pitch X.stride(0))."""
    _dev_check(X, out)
    c = ctx(X.device)
    check(lib().codae_row_sqnorm(c, p(X), X.stride(0), X.shape[0], E, p(out), stream()), c)


def rank_count(scores, Q, n, cc, qq, out_rank):
    """Ranks from a [Q, n + Q] matrix of dot products (columns n.. hold the true rows), cosine metric."""
    _dev_check(scores, cc, qq, out_rank)
    c = ctx(scores.device)
    check(lib().codae_rank_count(c, p(scores), scores.stride(0), Q, n, p(cc), p(qq), p(out_rank), stream()), c)


def swap_build(outfit, catalog, first_row, B, E, slot, io, inv_scale, out_x):
    _dev_check(outfit, catalog, out_x)
    c = ctx(catalog.device)
    check(lib().codae_swap_build(c, p(outfit), p(catalog), dt(catalog), catalog.stride(0), first_row, B, E, slot, io,
                                 inv_scale, p(out_x), dt(out_x), out_x.stride(0), stream()), c)


def swap_error_topk(outfit, catalog, first_row, B, E, slot, io, inv_scale, y, row_offset, k, out_score, out_idx, ws, allow=None,
                    exclude=None):
    """allow: uint8 [rows of catalog] or None; exclude: int64 [m] global indices or None (codae_swap_error_topk_filtered when
    either is given)."""
    _dev_check(outfit, catalog, y, out_score, out_idx, ws, allow, exclude)
    c = ctx(catalog.device)
    if allow is None and exclude is None:
        check(lib().codae_swap_error_topk(c, p(outfit), p(catalog), dt(catalog), catalog.stride(0), first_row, B, E, slot, io,
                                          inv_scale, p(y), y.stride(0), row_offset, k, p(out_score), p(out_idx), p(ws),
                                          ws.numel(), stream()), c)
        return
    ex, m = _n_exclude(exclude)
    check(lib().codae_swap_error_topk_filtered(c, p(outfit), p(catalog), dt(catalog), catalog.stride(0), first_row, B, E, slot,
                                               io, inv_scale, p(y), y.stride(0), row_offset, k, p(allow), p(ex), m, p(out_score),
                                               p(out_idx), p(ws), ws.numel(), stream()), c)


def swap_build_pairs(outfits, catalog, row_offset, candidates, pos, E, slot, io, inv_scale, out_x):
    """Rows of out_x: the pairs pos [B] (int64 indices into candidates [Q, m], global row ids) swapped into `slot` of their
    outfit (outfits [Q, io] f32)."""
    _dev_check(outfits, catalog, candidates, pos, out_x)
    c = ctx(catalog.device)
    Q, m = candidates.shape
    check(lib().codae_swap_build_pairs(c, p(outfits), outfits.stride(0), Q, p(catalog), dt(catalog), catalog.stride(0),
                                       catalog.shape[0], row_offset, p(candidates), m, p(pos), pos.numel(), E, slot, io, inv_scale,
                                       p(out_x), dt(out_x), out_x.stride(0), stream()), c)


def swap_error_pairs(outfits, catalog, row_offset, candidates, pos, E, slot, io, inv_scale, y, err):
    """err [Q m] f32: err[pos[b]] = swap error of reconstruction row b of y."""
    _dev_check(outfits, catalog, candidates, pos, y, err)
    c = ctx(catalog.device)
    Q, m = candidates.shape
    check(lib().codae_swap_error_pairs(c, p(outfits), outfits.stride(0), Q, p(catalog), dt(catalog), catalog.stride(0),
                                       catalog.shape[0], row_offset, p(candidates), m, p(pos), pos.numel(), E, slot, io, inv_scale,
                                       p(y), y.stride(0), p(err), stream()), c)


def swap_pairs_topk(err, candidates, k, out_score, out_idx):
    """Best k pairs per outfit by (error, candidate id): out_score [Q, k] f32, out_idx [Q, k] int64."""
    _dev_check(err, candidates, out_score, out_idx)
    c = ctx(err.device)
    Q, m = candidates.shape
    check(lib().codae_swap_pairs_topk(c, p(err), p(candidates), Q, m, k, p(out_score), p(out_idx), stream()), c)


def linear_engine(device, dtype, M, N, K):
    return lib().codae_linear_engine(ctx(device), dtype, M, N, K)
