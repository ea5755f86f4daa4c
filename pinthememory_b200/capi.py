"""ctypes binding of ``include/pinmem_b200.h`` -- the only way this package reaches the GPU.

There is no fallback: if ``_lib/libpinmem_b200.so`` is missing and cannot be built, or a call returns a
non-zero status, a ``RuntimeError`` is raised. Nothing here touches ``oracle/``.
"""
import ctypes
import os
import threading

import torch

from . import build as _build

PM_F32, PM_BF16 = 0, 1
WS_WORDS = 40  # PM_WS_WORDS
WS_HIST = 4    # PM_WS_HIST
WS_BAD = 2     # PM_WS_BAD

SEG_WS_WORDS = 4  # PM_SEG_WS_WORDS
SEG_WS_BAD = 2    # PM_SEG_WS_BAD

ABI_VERSION = 208  # PM_ABI_VERSION of include/pinmem_b200.h the argtypes below were written against

_c_p = ctypes.c_void_p
_c_i = ctypes.c_int
_c_f = ctypes.c_float
_c_d = ctypes.c_double

# name -> argtypes, exactly the prototypes of include/pinmem_b200.h
PROTOTYPES = {
    "pm_version": [],
    "pm_score_stride": [_c_i],
    "pm_colsoftmax_workspace_floats": [_c_i],
    "pm_read_fwd": [_c_p] * 8 + [_c_i] * 6 + [_c_p],
    "pm_colsoftmax": [_c_p] * 4 + [_c_i] * 2 + [_c_p],
    "pm_colsoftmax_apply": [_c_p] * 4 + [_c_i] * 2 + [_c_p],
    "pm_readloss_fwd": [_c_p, _c_p, _c_f] + [_c_i] * 6 + [_c_p] * 4,
    "pm_read_bwd": [_c_p] * 9 + [_c_i] * 6 + [_c_p],
    "pm_read_bwd_dM": [_c_p] * 5 + [_c_i] * 6 + [_c_p],
    "pm_read_planes": [],
    "pm_read_fwd_planes": [_c_p] * 8 + [_c_i] * 6 + [_c_p],
    "pm_read_bwd_planes": [_c_p] * 10 + [_c_i] * 6 + [_c_p],
    "pm_fold_weight_fwd": [_c_p] * 3 + [_c_i] * 3 + [_c_p],
    "pm_fold_weight_bwd": [_c_p] * 3 + [_c_i] * 3 + [_c_p],
    "pm_score_nhwc": [_c_p] * 3 + [_c_i] * 3 + [_c_p],
    "pm_rowsoftmax": [_c_p] * 3 + [_c_i] * 2 + [_c_p],
    "pm_write_reduce_fwd": [_c_p] * 3 + [_c_i] * 8 + [_c_p],
    "pm_update_aux_floats": [_c_i],
    "pm_update_fwd": [_c_p, _c_p, _c_f] + [_c_p] * 6 + [_c_i] * 2 + [_c_p],
    "pm_update_bwd": [_c_p] * 7 + [_c_f] + [_c_p] * 4 + [_c_i] * 2 + [_c_p],
    "pm_write_bwd": [_c_p] * 4 + [_c_i] * 8 + [_c_p],
    "pm_bn_stats": [_c_p] + [_c_i] * 4 + [_c_f] + [_c_p] * 4 + [_c_f, _c_p],
    "pm_bn_mask_words": [_c_i] * 3,
    "pm_bn_apply": [_c_p] * 8 + [_c_i] * 5 + [_c_p],
    "pm_bn_bwd_reduce": [_c_p] * 6 + [_c_i] + [_c_p] * 2 + [_c_i] * 4 + [_c_p],
    "pm_bn_bwd_scratch_bytes": [_c_i],
    "pm_bn_bwd_reduce_split": [_c_p] * 6 + [_c_i] + [_c_p] * 2 + [_c_i] * 4 + [_c_p] * 2,
    "pm_bn_bwd_rows_scratch_bytes": [_c_i] * 2,
    "pm_bn_bwd_reduce_rows": [_c_p] * 6 + [_c_i] + [_c_p] * 2 + [_c_i] * 4 + [_c_p] * 2,
    "pm_bn_bwd_apply": [_c_p] * 9 + [_c_i] * 2 + [_c_p] * 2 + [_c_i] * 4 + [_c_p],
    "pm_conv1x1_prep": [_c_p] + [_c_i] * 4 + [_c_p] * 3,
    "pm_conv1x1_prep_both": [_c_p, _c_i, _c_i, _c_i] + [_c_p] * 5 + [_c_i, _c_p],
    "pm_conv1x1_fwd": [_c_p] * 5 + [_c_i] * 6 + [_c_p],
    "pm_bn_eval_affine": [_c_p] * 4 + [_c_f, _c_i] + [_c_p] * 3,
    "pm_conv1x1_fwd_affine": [_c_p] * 6 + [_c_i] * 6 + [_c_p],
    "pm_conv1x1_wgrad_workspace_floats": [_c_i] * 5,
    "pm_conv1x1_wgrad": [_c_p] * 4 + [_c_i] * 6 + [_c_p],
    "pm_bn_finalize": [_c_p, _c_i, _c_d, _c_f] + [_c_p] * 4 + [_c_f, _c_p],
    "pm_conv1x1_dgrad_bnbwd": [_c_p] * 12 + [_c_i] * 7 + [_c_p],
    "pm_bn_apply_stats": [_c_p, _c_p, _c_d, _c_f] + [_c_p] * 5 + [_c_i] + [_c_p] * 4 + [_c_f, _c_p, _c_p] + [_c_i] * 4 + [_c_p],
    "pm_write_reduce_fwd8": [_c_p] * 3 + [_c_i] * 8 + [_c_p],
    "pm_write_bwd8": [_c_p] * 4 + [_c_i] * 8 + [_c_p],
    "pm_peer_buffer_bytes": [],
    "pm_update_fwd_peer": [_c_p, _c_i, _c_i, _c_p, _c_p, _c_p, _c_f] + [_c_p] * 6 + [_c_i] * 2 + [_c_p],
    "pm_update_bwd_peer": [_c_p, _c_i, _c_i, _c_p] + [_c_p] * 7 + [_c_f] + [_c_p] * 4 + [_c_i] * 2 + [_c_p],
    "pm_labels_pack": [_c_p, _c_i, ctypes.c_longlong, _c_i, _c_p, _c_p, _c_p],
    "pm_readloss_fwd8": [_c_p, _c_p, _c_f] + [_c_i] * 6 + [_c_p] * 4,
    "pm_memory_losses_fwd": [_c_p] * 3 + [_c_i] * 2 + [_c_p] * 4,
    "pm_memory_losses_bwd": [_c_p] * 6 + [_c_i] * 2 + [_c_p] * 4,
    "pm_seg_eval": [_c_p] + [_c_i] * 5 + [_c_p] + [_c_i] * 3 + [_c_p] * 5,
    "pm_upcat_fwd": [_c_p] * 3 + [_c_i] * 8 + [_c_p],
    "pm_upcat_bwd": [_c_p] * 2 + [_c_i] * 8 + [_c_p],
}
EXPORTED_SYMBOLS = sorted(list(PROTOTYPES) + ["pm_status_string"])

_lib = None
_lock = threading.Lock()


def library_path():
    return _build.LIB_PATH


def load():
    """Load (building first if the tree has no up-to-date library) and return the ctypes handle."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        # build() is a no-op when the library is newer than every source; a stale .so would otherwise be called
        # through argtypes written for newer prototypes (silent memory corruption, not an error)
        try:
            path = _build.build()
        except Exception:
            if not os.path.exists(_build.LIB_PATH):
                raise
            path = _build.LIB_PATH  # no compiler here (e.g. a run-only box): the version check below still guards
        lib = ctypes.CDLL(path)
        lib.pm_version.argtypes, lib.pm_version.restype = [], _c_i
        have = lib.pm_version()
        if have != ABI_VERSION:
            raise RuntimeError(f"pinmem_b200: {path} has ABI version {have}, this binding needs {ABI_VERSION}; "
                               "rebuild with `python -m pinthememory_b200.build --force`")
        for name, argtypes in PROTOTYPES.items():
            fn = getattr(lib, name)
            fn.argtypes = argtypes
            fn.restype = _c_i
        lib.pm_status_string.argtypes = [_c_i]
        lib.pm_status_string.restype = ctypes.c_char_p
        _lib = lib
    return _lib


def _check(code, what):
    if code != 0:
        msg = load().pm_status_string(code).decode()
        raise RuntimeError(f"pinmem_b200: {what} failed with status {code}: {msg}")


_tls = threading.local()


def _ptr(t):
    """Device address of a tensor argument; remembers its device so _call can refuse a cross-device launch."""
    if t is None:
        return None
    if t.is_cuda:
        devs = getattr(_tls, "devs", None)
        if devs is None:
            devs = _tls.devs = set()
        devs.add(t.device.index)
    return t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _check_devices(name):
    """Every kernel launches on the CURRENT device and its current stream, so a tensor living on another GPU would be
    dereferenced on the wrong one (an illegal address at best): refuse instead. Wrap the call in
    ``torch.cuda.device(tensor.device)`` (or ``torch.cuda.set_device``) when the module is not on the current device."""
    devs = getattr(_tls, "devs", None)
    if not devs:
        return
    cur = torch.cuda.current_device()
    bad = [d for d in devs if d != cur]
    devs.clear()
    if bad:
        raise RuntimeError(f"pinmem_b200: {name} got tensors on cuda:{bad[0]} while the current device is cuda:{cur}; "
                           "launch under torch.cuda.device(...) of the tensors' device")


def dtype_code(t):
    if t.dtype == torch.float32:
        return PM_F32
    if t.dtype == torch.bfloat16:
        return PM_BF16
    raise RuntimeError(f"pinmem_b200: feature dtype must be float32 or bfloat16, got {t.dtype}")


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("pinmem_b200 has no CPU path: every tensor must live on a CUDA device")


def _f32c(t, what):
    if t.dtype != torch.float32 or not t.is_contiguous():
        raise RuntimeError(f"pinmem_b200: {what} must be a contiguous float32 tensor")
    return t


def score_stride(K):
    return load().pm_score_stride(int(K))


# ------------------------------------------------------------------------------- launch accounting
# bench.py counts the kernels launched inside its timed region and (optionally) brackets every C-ABI call
# with CUDA events on the launching stream to get per-kernel durations live.

LAUNCHES = 0
_KERNELS_PER_CALL = {"pm_conv1x1_dgrad_bnbwd": 2, "pm_colsoftmax": 3, "pm_colsoftmax_apply": 1, "pm_read_bwd": 2, "pm_read_bwd_planes": 2, "pm_conv1x1_wgrad": 2}
PLANES = 32  # PM_PLANES: score planes appended to q in the score-plane read
_timing = None  # name -> list of (start_event, end_event) when enabled


def enable_kernel_timing(on=True):
    global _timing
    _timing = {} if on else None


def kernel_timings_ms():
    """name -> list of per-call durations (ms). Synchronises."""
    if _timing is None:
        return {}
    torch.cuda.synchronize()
    return {k: [a.elapsed_time(b) for a, b in v] for k, v in _timing.items()}


def reset_counters():
    global LAUNCHES
    LAUNCHES = 0
    if _timing is not None:
        _timing.clear()


def _call(name, *args):
    global LAUNCHES
    fn = getattr(load(), name)
    _check_devices(name)
    if _timing is None:
        code = fn(*args)
    else:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        code = fn(*args)
        b.record()
        _timing.setdefault(name, []).append((a, b))
    LAUNCHES += _KERNELS_PER_CALL.get(name, 1)
    _check(code, name)


# --------------------------------------------------------------------------------------------- calls


def planes_ok(x):
    """The score-plane read runs only on the pipelined kernels: 16-byte rows and pointers."""
    hw = x.shape[2] * x.shape[3]
    return x.is_cuda and hw % (4 if x.dtype == torch.float32 else 8) == 0 and x.data_ptr() % 16 == 0


def read_fwd(x, M, gumbel_m, u, s, score_m, K, gumbel_q=None, col_partials=None, planes=False):
    B, C, h, w = x.shape
    _call("pm_read_fwd_planes" if planes else "pm_read_fwd", _ptr(x), _ptr(M), _ptr(gumbel_m), _ptr(gumbel_q), _ptr(u), _ptr(s), _ptr(score_m),
          _ptr(col_partials), B, C, h, w, K, dtype_code(x), _stream())


def colsoftmax_apply(s, gumbel_q, col_partials, score_q, N, K):
    _call("pm_colsoftmax_apply", _ptr(s), _ptr(gumbel_q), _ptr(col_partials), _ptr(score_q), N, K, _stream())


def colsoftmax(s, gumbel_q, score_q, workspace, N, K):
    _call("pm_colsoftmax", _ptr(s), _ptr(gumbel_q), _ptr(score_q), _ptr(workspace), N, K, _stream())


def colsoftmax_workspace_floats(K):
    return load().pm_colsoftmax_workspace_floats(int(K))


def readloss_fwd(s, labels, temperature, B, h, w, K, ds_rl, ws, out):
    Hm, Wm = labels.shape[1], labels.shape[2]
    _call("pm_readloss_fwd", _ptr(s), _ptr(labels), float(temperature), B, h, w, Hm, Wm, K, _ptr(ds_rl),
                                  _ptr(ws), _ptr(out), _stream())


def read_bwd(du, x, M, score_m, ds_rl, g_loss, rl_out, dx, ds, K, planes=False, dx_add=None):
    """``dx_add`` (score-plane read only): a second gradient of x summed into dx by the kernel."""
    B, C, h, w = x.shape
    if planes:
        _call("pm_read_bwd_planes", _ptr(du), _ptr(x), _ptr(M), _ptr(score_m), _ptr(ds_rl), _ptr(g_loss), _ptr(rl_out),
              _ptr(dx), _ptr(dx_add), _ptr(ds), B, C, h, w, K, dtype_code(x), _stream())
        return
    if dx_add is not None:
        raise RuntimeError("pinmem_b200: dx_add is only supported by the score-plane read backward")
    _call("pm_read_bwd", _ptr(du), _ptr(x), _ptr(M), _ptr(score_m), _ptr(ds_rl), _ptr(g_loss), _ptr(rl_out),
          _ptr(dx), _ptr(ds), B, C, h, w, K, dtype_code(x), _stream())


def read_bwd_dM(du, x, score_m, ds, dM, K):
    B, C, h, w = x.shape
    _call("pm_read_bwd_dM", _ptr(du), _ptr(x), _ptr(score_m), _ptr(ds), _ptr(dM), B, C, h, w, K,
                                 dtype_code(x), _stream())


def fold_weight_fwd(W, M, Wp, Co, C, K):
    _call("pm_fold_weight_fwd", _ptr(W), _ptr(M), _ptr(Wp), Co, C, K, _stream())


def fold_weight_bwd(dWp, M, dW, Co, C, K):
    _call("pm_fold_weight_bwd", _ptr(dWp), _ptr(M), _ptr(dW), Co, C, K, _stream())


def score_nhwc(q, M, s, N, C, K):
    _call("pm_score_nhwc", _ptr(q), _ptr(M), _ptr(s), N, C, K, _stream())


def rowsoftmax(s, gumbel_m, score_m, N, K):
    _call("pm_rowsoftmax", _ptr(s), _ptr(gumbel_m), _ptr(score_m), N, K, _stream())


def write_reduce_fwd(f, labels, SD, K):
    """labels: int64 class ids, or the packed uint8 map of labels_pack (class K = ignore)."""
    B, C, h, w = f.shape
    Hm, Wm = labels.shape[1], labels.shape[2]
    _call("pm_write_reduce_fwd8" if labels.dtype == torch.uint8 else "pm_write_reduce_fwd", _ptr(f), _ptr(labels), _ptr(SD), B, C, h, w, Hm, Wm, K, dtype_code(f),
                                      _stream())


def update_aux_floats(K):
    return load().pm_update_aux_floats(int(K))


def update_aux(device, K):
    """Zeroed scratch for one pm_update_fwd / pm_update_bwd call."""
    return torch.zeros(update_aux_floats(K), dtype=torch.float32, device=device)


def update_fwd(SD, M_old, momentum, W, b, M_new, losses, saved, C, K, aux=None):
    if aux is None:
        aux = update_aux(SD.device, K)
    _call("pm_update_fwd", _ptr(SD), _ptr(M_old), float(momentum), _ptr(W), _ptr(b), _ptr(M_new),
          _ptr(losses), _ptr(saved), _ptr(aux), C, K, _stream())


def update_bwd(dM_new, g_div, g_cls, M_new, saved, W, b, momentum, dS, dW, db, C, K):
    _call("pm_update_bwd", _ptr(dM_new), _ptr(g_div), _ptr(g_cls), _ptr(M_new), _ptr(saved), _ptr(W), _ptr(b),
          float(momentum), _ptr(dS), _ptr(dW), _ptr(db), _ptr(update_aux(M_new.device, K)), C, K, _stream())


def write_bwd(dS, f, labels, df, K):
    B, C, h, w = f.shape
    Hm, Wm = labels.shape[1], labels.shape[2]
    _call("pm_write_bwd8" if labels.dtype == torch.uint8 else "pm_write_bwd", _ptr(dS), _ptr(f), _ptr(labels), _ptr(df), B, C, h, w, Hm, Wm, K, dtype_code(f),
                               _stream())


def bn_stats(x, eps, mean, invstd, running_mean, running_var, momentum):
    B, C, h, w = x.shape
    _call("pm_bn_stats", _ptr(x), B, C, h * w, dtype_code(x), float(eps), _ptr(mean), _ptr(invstd), _ptr(running_mean),
          _ptr(running_var), float(momentum), _stream())


def bn_mask_words(B, C, hw):
    return load().pm_bn_mask_words(int(B), int(C), int(hw))


def bn_apply(x, mean, invstd, gamma, beta, residual, y, relu, relu_mask=None):
    B, C, h, w = x.shape
    _call("pm_bn_apply", _ptr(x), _ptr(mean), _ptr(invstd), _ptr(gamma), _ptr(beta), _ptr(residual), _ptr(y),
          _ptr(relu_mask), int(relu), B, C, h * w, dtype_code(x), _stream())


_BN_ROWS_SCRATCH = {}  # (device, stream, B, C) -> zero-initialised scratch of pm_bn_bwd_reduce_rows (self-cleaning counters)


def _bn_rows_scratch(x, B, C):
    st = torch.cuda.current_stream(x.device)
    key = (x.device.index, st.cuda_stream, B, C)
    buf = _BN_ROWS_SCRATCH.get(key)
    if buf is None:
        # (allocated inside a graph capture the fill becomes a memset node that re-zeroes on every replay: harmless, and this
        # cache keeps the buffer alive as long as the graph)
        buf = torch.zeros(load().pm_bn_bwd_rows_scratch_bytes(B, C) // 8 + 1, dtype=torch.float64, device=x.device)
        _BN_ROWS_SCRATCH[key] = buf
    return buf


def bn_bwd_reduce(dy, y, relu_mask, x, mean, invstd, relu, dgamma, dbeta):
    B, C, h, w = x.shape
    if not os.environ.get("PINMEM_B200_BN_REDUCE_PER_CHANNEL"):  # one CTA per (image, channel) row: 48 -> ~30 us at cfg 2
        _call("pm_bn_bwd_reduce_rows", _ptr(dy), _ptr(y), _ptr(relu_mask), _ptr(x), _ptr(mean), _ptr(invstd), int(relu),
              _ptr(dgamma), _ptr(dbeta), B, C, h * w, dtype_code(x), _ptr(_bn_rows_scratch(x, B, C)), _stream())
        return
    if os.environ.get("PINMEM_B200_BN_SPLIT"):   # measured 55.7 us vs 51 us unsplit at cfg 2: off by default (A/B switch)
        scratch = torch.zeros(load().pm_bn_bwd_scratch_bytes(C) // 8 + 1, dtype=torch.float64, device=x.device)
        _call("pm_bn_bwd_reduce_split", _ptr(dy), _ptr(y), _ptr(relu_mask), _ptr(x), _ptr(mean), _ptr(invstd), int(relu),
              _ptr(dgamma), _ptr(dbeta), B, C, h * w, dtype_code(x), _ptr(scratch), _stream())
        return
    _call("pm_bn_bwd_reduce", _ptr(dy), _ptr(y), _ptr(relu_mask), _ptr(x), _ptr(mean), _ptr(invstd), int(relu),
          _ptr(dgamma), _ptr(dbeta), B, C, h * w, dtype_code(x), _stream())


def bn_bwd_apply(dy, y, relu_mask, x, mean, invstd, gamma, dgamma, dbeta, relu, training, dx, dres):
    B, C, h, w = x.shape
    _call("pm_bn_bwd_apply", _ptr(dy), _ptr(y), _ptr(relu_mask), _ptr(x), _ptr(mean), _ptr(invstd), _ptr(gamma),
          _ptr(dgamma), _ptr(dbeta), int(relu), int(training), _ptr(dx), _ptr(dres), B, C, h * w, dtype_code(x),
          _stream())


# ------------------------------------------------------------------------ 1x1 convolutions (csrc/pm_gemm.cu)


def conv1x1_prep(W2d, transpose, dtype):
    """W2d fp32 [R,S] -> operand A = W2d (transpose False: M=R, K=S) or W2d^T (True: M=S, K=R), zero-padded to a multiple
    of 128 rows; fp32 returns (A_hi, A_lo) fp32, bf16 returns (A, None)."""
    R, S = W2d.shape
    M, K = (S, R) if transpose else (R, S)
    Mpad = (M + 127) // 128 * 128
    W2d = _f32c(W2d, "weight")
    hi = torch.empty(Mpad, K, dtype=dtype, device=W2d.device)
    lo = torch.empty(Mpad, K, dtype=dtype, device=W2d.device) if dtype == torch.float32 else None
    _call("pm_conv1x1_prep", _ptr(W2d), M, K, int(bool(transpose)), PM_F32 if dtype == torch.float32 else PM_BF16,
          _ptr(hi), _ptr(lo), _stream())
    return hi, lo


def conv1x1_prep_both(W2d, dtype, zero=None):
    """((A_hi, A_lo), (At_hi, At_lo)): conv1x1_prep(W2d, False) and conv1x1_prep(W2d, True) from one launch, which also
    clears the float64 buffer ``zero`` (the BatchNorm statistics the forward GEMM's epilogue adds into)."""
    R, S = W2d.shape
    W2d = _f32c(W2d, "weight")
    f32 = dtype == torch.float32
    hi = torch.empty((R + 127) // 128 * 128, S, dtype=dtype, device=W2d.device)
    lo = torch.empty_like(hi) if f32 else None
    hiT = torch.empty((S + 127) // 128 * 128, R, dtype=dtype, device=W2d.device)
    loT = torch.empty_like(hiT) if f32 else None
    if zero is not None and (zero.dtype != torch.float64 or not zero.is_contiguous()):
        raise ValueError("conv1x1_prep_both: `zero` must be a contiguous float64 tensor")
    _call("pm_conv1x1_prep_both", _ptr(W2d), R, S, PM_F32 if f32 else PM_BF16, _ptr(hi), _ptr(lo), _ptr(hiT), _ptr(loT),
          _ptr(zero), 0 if zero is None else zero.numel(), _stream())
    return (hi, lo), (hiT, loT)


def conv1x1_ok(x, M, K):
    """Shapes/alignments the tcgen05 GEMMs take (everything the module produces on aligned feature maps)."""
    hw = x.shape[2] * x.shape[3]
    esz = 4 if x.dtype == torch.float32 else 2
    return (x.is_cuda and x.dtype in (torch.float32, torch.bfloat16) and (hw * esz) % 16 == 0 and x.data_ptr() % 16 == 0
            and K % (8 if esz == 4 else 16) == 0 and M % 32 == 0 and M <= 512 and K % 32 == 0 and K <= 1024)


def conv1x1_fwd(x, A_hi, A_lo, M, y=None, stats=None, accumulate=False):
    """y[b] (M x hw) (+)= A (M x K) . x[b] (K x hw); stats: zeroed double[2M] receiving per-row sum / sum of squares."""
    B, K, h, w = x.shape
    if y is None:
        y = torch.empty(B, M, h, w, dtype=x.dtype, device=x.device)
    _call("pm_conv1x1_fwd", _ptr(x), _ptr(A_hi), _ptr(A_lo), _ptr(y), _ptr(stats), B, K, M, h * w, int(bool(accumulate)),
          dtype_code(x), _stream())
    return y


def conv1x1_dgrad_bnbwd(dy, z, A_hi, A_lo, M, mean, invstd, gamma, dgamma, dbeta, beta, relu, training):
    """(dx [B,M,h,w], dz [B,K,h,w]): input gradient of conv1x1 -> BatchNorm (-> ReLU) with the BatchNorm backward formed in
    the GEMM's operand path; dz is stored for the weight-gradient GEMM (fp32 only)."""
    B, K, h, w = dy.shape
    dx = torch.empty(B, M, h, w, dtype=dy.dtype, device=dy.device)
    dz = torch.empty_like(dy)
    _call("pm_conv1x1_dgrad_bnbwd", _ptr(dy), _ptr(z), _ptr(A_hi), _ptr(A_lo), _ptr(dx), _ptr(dz), _ptr(mean), _ptr(invstd),
          _ptr(gamma), _ptr(beta), _ptr(dgamma), _ptr(dbeta), int(bool(relu)), int(bool(training)), B, K, M, h * w,
          dtype_code(dy), _stream())
    return dx, dz


def bn_eval_affine(gamma, beta, running_mean, running_var, eps):
    """Eval-mode BatchNorm2d as (scale, shift) fp32 [C] for pm_conv1x1_fwd_affine."""
    C = gamma.shape[0]
    scale = torch.empty(C, dtype=torch.float32, device=gamma.device)
    shift = torch.empty(C, dtype=torch.float32, device=gamma.device)
    _call("pm_bn_eval_affine", _ptr(gamma), _ptr(beta), _ptr(running_mean), _ptr(running_var), float(eps), C, _ptr(scale),
          _ptr(shift), _stream())
    return scale, shift


def conv1x1_fwd_affine(x, A_hi, A_lo, M, scale, shift, relu):
    """y[b] = [relu](scale[m] * (A . x[b]) + shift[m]) -- convolution + eval-mode BatchNorm (+ ReLU) in one kernel."""
    B, K, h, w = x.shape
    y = torch.empty(B, M, h, w, dtype=x.dtype, device=x.device)
    _call("pm_conv1x1_fwd_affine", _ptr(x), _ptr(A_hi), _ptr(A_lo), _ptr(y), _ptr(scale), _ptr(shift), int(bool(relu)), B, K, M,
          h * w, dtype_code(x), _stream())
    return y


def conv1x1_wgrad(dy, x, dW=None, accumulate=False):
    """dW [M,N] fp32 (+)= sum_b dy[b] (M x hw) . x[b]^T (hw x N)."""
    B, M, h, w = dy.shape
    N = x.shape[1]
    if dW is None:
        dW = torch.empty(M, N, dtype=torch.float32, device=x.device)
    nws = load().pm_conv1x1_wgrad_workspace_floats(B, M, N, h * w, dtype_code(x))
    ws = torch.empty(nws, dtype=torch.float32, device=x.device)
    _call("pm_conv1x1_wgrad", _ptr(dy), _ptr(x), _ptr(ws), _ptr(dW), B, M, N, h * w, int(bool(accumulate)), dtype_code(x),
          _stream())
    return dW


def bn_apply_stats(x, stats, count, eps, gamma, beta, residual, y, relu, mean_out, invstd_out, running_mean, running_var,
                   momentum, relu_mask=None, count_dev=None, num_batches_tracked=None):
    """Normalise pass with the batch statistics finalised in-kernel from the GEMM epilogue's fp64 sums (``count_dev``: a
    float64 device scalar that replaces ``count`` -- the all-reduced global count of a SyncBatchNorm)."""
    B, C, h, w = x.shape
    _call("pm_bn_apply_stats", _ptr(x), _ptr(stats), float(count), float(eps), _ptr(gamma), _ptr(beta), _ptr(residual), _ptr(y),
          _ptr(relu_mask), int(bool(relu)), _ptr(mean_out), _ptr(invstd_out), _ptr(running_mean), _ptr(running_var),
          float(momentum), _ptr(count_dev), _ptr(num_batches_tracked), B, C, h * w, dtype_code(x), _stream())


def bn_finalize(stats, C, count, eps, mean, invstd, running_mean, running_var, momentum):
    _call("pm_bn_finalize", _ptr(stats), C, float(count), float(eps), _ptr(mean), _ptr(invstd), _ptr(running_mean),
          _ptr(running_var), float(momentum), _stream())


# ------------------------------------------------------------ stand-alone write losses (csrc/pm_losses.cu)


def memory_losses_fwd(mem, W, b, out, gram, prob):
    K, C = mem.shape
    _call("pm_memory_losses_fwd", _ptr(mem), _ptr(W), _ptr(b), K, C, _ptr(out), _ptr(gram), _ptr(prob), _stream())


def memory_losses_bwd(mem, W, gram, prob, g_div, g_cls, dmem, dW, db):
    K, C = mem.shape
    _call("pm_memory_losses_bwd", _ptr(mem), _ptr(W), _ptr(gram), _ptr(prob), _ptr(g_div), _ptr(g_cls), K, C, _ptr(dmem),
          _ptr(dW), _ptr(db), _stream())


# --------------------------------------------------------------------- packed labels (csrc/pm_labels.cu)


def labels_pack(labels, K, ws):
    """int64 | uint8 labels -> uint8 class map (K = ignore); histogram and bad-label count into the zeroed ws."""
    lab8 = torch.empty(labels.shape, dtype=torch.uint8, device=labels.device)
    _call("pm_labels_pack", _ptr(labels), int(labels.dtype == torch.uint8), labels.numel(), int(K), _ptr(lab8), _ptr(ws),
          _stream())
    return lab8


def readloss_fwd8(s, lab8, temperature, B, h, w, K, ds_rl, ws, out):
    Hm, Wm = lab8.shape[1], lab8.shape[2]
    _call("pm_readloss_fwd8", _ptr(s), _ptr(lab8), float(temperature), B, h, w, Hm, Wm, K, _ptr(ds_rl), _ptr(ws), _ptr(out),
          _stream())


def seg_eval(logits, labels, confusion, pred, ws, out):
    """Up-sample + argmax + cross-entropy + confusion increments in one label pass (csrc/pm_segeval.cu)."""
    B, K, h, w = logits.shape
    Hm, Wm = labels.shape[1], labels.shape[2]
    _call("pm_seg_eval", _ptr(logits), dtype_code(logits), B, K, h, w, _ptr(labels), int(labels.dtype == torch.uint8), Hm, Wm,
          _ptr(confusion), _ptr(pred), _ptr(ws), _ptr(out), _stream())


def upcat_fwd(fine, coarse, out):
    """out [B,Cf+Cc,H,W] = cat(fine, bilinear up-sample of coarse, align_corners=True) in one kernel (csrc/pm_upcat.cu)."""
    B, Cf, H, W = fine.shape
    _, Cc, h, w = coarse.shape
    _call("pm_upcat_fwd", _ptr(fine) if Cf else None, _ptr(coarse), _ptr(out), dtype_code(coarse), B, Cf, Cc, h, w, H, W,
          _stream())


def upcat_bwd(g, d_coarse, Cf):
    """d_coarse [B,Cc,h,w] from the planes [Cf,Cf+Cc) of the contiguous gradient g [B,Cf+Cc,H,W], read in place."""
    B, _, H, W = g.shape
    _, Cc, h, w = d_coarse.shape
    _call("pm_upcat_bwd", _ptr(g), _ptr(d_coarse), dtype_code(g), B, Cf, Cc, h, w, H, W, _stream())


def readloss(s, labels, temperature, B, h, w, K, ds_rl, ws, out):
    """Read loss on int64 | uint8 labels: one label pass (pack + histogram + bad-label count) and the second-generation
    kernel for K <= 19, the first kernel (int64 labels, any K <= 31) otherwise or with PINMEM_B200_READLOSS_V1 set."""
    if K <= 19 and not os.environ.get("PINMEM_B200_READLOSS_V1"):
        lab8 = labels_pack(labels, K, ws)
        readloss_fwd8(s, lab8, temperature, B, h, w, K, ds_rl, ws, out)
        return lab8
    readloss_fwd(s, labels if labels.dtype == torch.int64 else labels.to(torch.int64), temperature, B, h, w, K, ds_rl, ws, out)
    return None


# ------------------------------------- sharded update with the exchange fused over peer memory (csrc/pm_write.cu)

PEER_DS_OFF, PEER_FLAG_OFF, PEER_BYTES = 36864, 73728, 131072  # PM_PEER_* of the header


def update_fwd_peer(peer, SD_sum, M_old, momentum, W, b, M_new, losses, saved, C, K, aux=None):
    if aux is None:
        aux = update_aux(M_old.device, K)
    _call("pm_update_fwd_peer", peer.bufs_dev, peer.rank, peer.world_size, _ptr(peer.epochs[0:1]), _ptr(SD_sum), _ptr(M_old),
          float(momentum), _ptr(W), _ptr(b), _ptr(M_new), _ptr(losses), _ptr(saved), _ptr(aux), C, K, _stream())


def update_bwd_peer(peer, dM_new, g_div, g_cls, M_new, saved, W, b, momentum, dS, dW, db, C, K):
    _call("pm_update_bwd_peer", peer.bufs_dev, peer.rank, peer.world_size, _ptr(peer.epochs[1:2]), _ptr(dM_new), _ptr(g_div),
          _ptr(g_cls), _ptr(M_new), _ptr(saved), _ptr(W), _ptr(b), float(momentum), _ptr(dS), _ptr(dW), _ptr(db),
          _ptr(update_aux(M_new.device, K)), C, K, _stream())
