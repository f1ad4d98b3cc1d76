"""ctypes binding of the C-ABI kernel library (``include/frl_b200.h``).

There is no fallback: if ``csrc/libfrl_b200.so`` is missing or a launch fails this module
raises.  ``python __graft_entry__.py build`` (or ``make -C csrc``) produces the library in-tree.
"""
import ctypes as C
import os
import subprocess
from typing import Optional, Sequence

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC_DIR = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(CSRC_DIR, "libfrl_b200.so")

F32, BF16, U8, I64 = 0, 1, 2, 3
LOSS_MSE, LOSS_CE = 0, 1
MAX_TASKS = 8

_DTYPE_CODE = {torch.float32: F32, torch.bfloat16: BF16, torch.uint8: U8, torch.bool: U8,
               torch.int64: I64}


class NativeLibraryError(RuntimeError):
    pass


class TaskDesc(C.Structure):
    """Mirror of ``frl_task_desc``."""
    _fields_ = [
        ("kind", C.c_int32), ("out_dtype", C.c_int32), ("tgt_dtype", C.c_int32),
        ("ignore_index", C.c_int32),
        ("out", C.c_void_p), ("tgt", C.c_void_p), ("mask", C.c_void_p), ("dout", C.c_void_p),
        ("rows", C.c_int64), ("cols", C.c_int64), ("mask_inner", C.c_int64),
        ("weight", C.c_float), ("_pad", C.c_float),
    ]


class GradSeg(C.Structure):
    """Mirror of ``frl_grad_seg``."""
    _fields_ = [("g", C.c_void_p), ("arena_off", C.c_int64), ("numel", C.c_int64),
                ("g_dtype", C.c_int32), ("_pad", C.c_int32)]


# name -> (restype, argtypes); every name here must be declared in include/frl_b200.h
_vp, _i, _i64, _f, _d = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double
SIGNATURES = {
    "frl_abi_version": (_i, []),
    "frl_last_error": (C.c_char_p, []),
    "frl_launch_count": (C.c_uint64, []),
    "frl_launch_count_reset": (None, []),
    "frl_device_sm_count": (_i, []),
    "frl_device_arch": (_i, []),
    "frl_sgd_momentum": (_i, [_vp, _vp, _vp, _vp, _i64, _d, _d, _d, _d, _d, _vp, _vp, _i, _i, _vp]),
    "frl_adam": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _d, _d, _d, _d, _d, _i64, _d, _vp, _vp, _i, _vp]),
    "frl_adamw": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _d, _d, _d, _d, _d, _i64, _d, _vp, _vp, _i, _vp]),
    "frl_rmsprop": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _d, _d, _d, _d, _d, _d, _vp, _vp, _i, _vp]),
    "frl_mt_tile_elems": (_i64, []),
    "frl_flatten_grads": (_i, [_vp, _vp, _vp, _i64, _vp, _i, _d, _vp]),
    "frl_sgd_momentum_mt": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _d, _d, _d, _d, _d, _vp, _vp, _i, _vp]),
    "frl_adam_mt": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _d, _d, _d, _d, _d, _i64, _d, _vp, _vp, _vp]),
    "frl_adamw_mt": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _d, _d, _d, _d, _d, _i64, _d, _vp, _vp, _vp]),
    "frl_rmsprop_mt": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _d, _d, _d, _d, _d, _d, _vp, _vp, _vp]),
    "frl_reduce_scratch_bytes": (_i64, []),
    "frl_grad_sumsq_clip": (_i, [_vp, _i64, _i, _f, _f, _vp, _vp, _vp]),
    "frl_criteria_scratch_bytes": (_i64, [_i]),
    "frl_criteria_forward": (_i, [C.POINTER(TaskDesc), _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "frl_criteria_backward": (_i, [C.POINTER(TaskDesc), _i, _vp, _vp, _vp, _vp]),
    "frl_preproc_affine": (_i, [_vp, _i, _vp, _i, _i64, _i64, _i64, _vp, _vp, _vp]),
    "frl_cast_scale": (_i, [_vp, _i, _vp, _i, _i64, _f, _vp]),
    "frl_colsum_scratch_bytes": (_i64, [_i64, _i64]),
    "frl_colsum": (_i, [_vp, _i, _i64, _i64, _vp, _i, _i, _vp, _vp]),
    "frl_drelu_colsum": (_i, [_vp, _vp, _vp, _i, _i64, _i64, _vp, _i, _i, _vp, _vp]),
    "frl_gather_rows": (_i, [_vp, _i64, _vp, _vp, _i64, _i64, _i, _vp]),
    "frl_gather_rows_tma": (_i, [_vp, _i64, _vp, _vp, _i64, _i64, _i, _vp]),
    "frl_gather_window_rows": (_i, [_vp, _vp, _i, _vp, _vp, _i64, _i64, _vp]),
    "frl_gather_pool_create": (_vp, [_i]),
    "frl_gather_pool_destroy": (None, [_vp]),
    "frl_gather_pool_threads": (_i, [_vp]),
    "frl_gather_pool_submit": (_i64, [_vp, _vp, _i64, _vp, _vp, _i64, _i64]),
    "frl_gather_pool_submit_f32_to_bf16": (_i64, [_vp, _vp, _i64, _vp, _vp, _i64, _i64]),
    "frl_gather_pool_wait": (_i, [_vp, _i64]),
    "frl_nvls_sgd": (_i, [_vp, _vp, _vp, _vp, _i64, _i, _i, _vp, _i, _vp, _i, _d, _d, _d, _d, _d, _vp, _i, _i, _i, _vp]),
    "frl_nvls_adam": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _vp, _i, _vp, _i, _d, _d, _d, _d, _d,
                           _i64, _d, _vp, _i, _i, _vp]),
    "frl_nvls_adamw": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _vp, _i, _vp, _i, _d, _d, _d, _d, _d,
                            _i64, _d, _vp, _i, _i, _vp]),
    "frl_nvls_rmsprop": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _vp, _i, _vp, _i, _d, _d, _d, _d, _d, _d,
                              _vp, _i, _i, _vp]),
    "frl_nvls_barrier": (_i, [_vp, _i, _i, _i, _vp]),
}

_lib: Optional[C.CDLL] = None


def build(verbose: bool = False) -> str:
    """Compile the library in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC_DIR, "-j8"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout)
        print(res.stderr)
    if res.returncode != 0:
        raise NativeLibraryError("building libfrl_b200.so failed:\n" + res.stderr[-4000:])
    return LIB_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryError(
                f"{LIB_PATH} is missing: the sm_100a kernel library has not been built "
                "(run `python __graft_entry__.py build` or `make -C <pkg>/csrc`). "
                "There is no fallback path.")
        handle = C.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(handle, name)        # AttributeError if the .so is stale
            fn.restype = restype
            fn.argtypes = argtypes
        if handle.frl_abi_version() != 1:
            raise NativeLibraryError("libfrl_b200.so ABI version mismatch; rebuild")
        _lib = handle
    return _lib


def is_available() -> bool:
    return os.path.exists(LIB_PATH)


def _check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().frl_last_error().decode("utf-8", "replace")
        raise NativeLibraryError(f"{what} failed (rc={rc}): {msg}")


def dtype_code(dt: torch.dtype) -> int:
    try:
        return _DTYPE_CODE[dt]
    except KeyError:
        raise NativeLibraryError(f"dtype {dt} has no kernel path") from None


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def launch_count() -> int:
    return int(lib().frl_launch_count())


def launch_count_reset() -> None:
    lib().frl_launch_count_reset()


# ---- K2 -------------------------------------------------------------------------------------

def sgd_momentum(p, g, buf, p_lp, n, *, lr, mu, dampening, wd, grad_scale=1.0,
                 grad_scale_dev=None, first_step=False, dyn=None) -> None:
    _check(lib().frl_sgd_momentum(_ptr(p), _ptr(g), _ptr(buf), _ptr(p_lp), n, lr, mu, dampening,
                                  wd, grad_scale, _ptr(grad_scale_dev), _ptr(dyn), int(first_step),
                                  dtype_code(g.dtype), _stream()), "frl_sgd_momentum")


def adam(p, g, m, v, vmax, p_lp, n, *, lr, beta1, beta2, eps, wd, step, grad_scale=1.0,
         grad_scale_dev=None, dyn=None) -> None:
    _check(lib().frl_adam(_ptr(p), _ptr(g), _ptr(m), _ptr(v), _ptr(vmax), _ptr(p_lp), n, lr,
                          beta1, beta2, eps, wd, step, grad_scale, _ptr(grad_scale_dev), _ptr(dyn),
                          dtype_code(g.dtype), _stream()), "frl_adam")


def adamw(p, g, m, v, vmax, p_lp, n, *, lr, beta1, beta2, eps, wd, step, grad_scale=1.0,
          grad_scale_dev=None, dyn=None) -> None:
    """``adam`` with decoupled weight decay (torch.optim.AdamW): p *= 1 - lr*wd, g not decayed."""
    _check(lib().frl_adamw(_ptr(p), _ptr(g), _ptr(m), _ptr(v), _ptr(vmax), _ptr(p_lp), n, lr,
                           beta1, beta2, eps, wd, step, grad_scale, _ptr(grad_scale_dev), _ptr(dyn),
                           dtype_code(g.dtype), _stream()), "frl_adamw")


def rmsprop(p, g, sq, buf, p_lp, n, *, lr, alpha, eps, wd, mu, grad_scale=1.0,
            grad_scale_dev=None, dyn=None) -> None:
    _check(lib().frl_rmsprop(_ptr(p), _ptr(g), _ptr(sq), _ptr(buf), _ptr(p_lp), n, lr, alpha,
                             eps, wd, mu, grad_scale, _ptr(grad_scale_dev), _ptr(dyn),
                             dtype_code(g.dtype), _stream()), "frl_rmsprop")


# ---- K2-mt / K1: multi-tensor forms (gradients read where autograd left them) ---------------------

def mt_tile_elems() -> int:
    return int(lib().frl_mt_tile_elems())


def flatten_grads(table, arena_grad, *, scale: float = 1.0) -> None:
    """arena_grad[seg.arena_off + i] = cast(seg.g[i] * scale) for every segment of ``table``
    (a ``multi_tensor.GradSegTable`` whose device copy is current): one launch."""
    _check(lib().frl_flatten_grads(table.segs_dev_ptr, table.prefix_dev_ptr, table.tile_seg_dev_ptr, table.n_tiles,
                                   _ptr(arena_grad), dtype_code(arena_grad.dtype), scale, _stream()),
           "frl_flatten_grads")


def sgd_momentum_mt(p, buf, p_lp, table, *, lr, mu, dampening, wd, grad_scale=1.0, grad_scale_dev=None,
                    first_step=False, dyn=None) -> None:
    _check(lib().frl_sgd_momentum_mt(_ptr(p), _ptr(buf), _ptr(p_lp), table.segs_dev_ptr, table.prefix_dev_ptr,
                                     table.tile_seg_dev_ptr, table.n_tiles, lr, mu, dampening, wd, grad_scale,
                                     _ptr(grad_scale_dev), _ptr(dyn), int(first_step), _stream()),
           "frl_sgd_momentum_mt")


def adam_mt(p, m, v, vmax, p_lp, table, *, lr, beta1, beta2, eps, wd, step, grad_scale=1.0,
            grad_scale_dev=None, dyn=None) -> None:
    _check(lib().frl_adam_mt(_ptr(p), _ptr(m), _ptr(v), _ptr(vmax), _ptr(p_lp), table.segs_dev_ptr,
                             table.prefix_dev_ptr, table.tile_seg_dev_ptr, table.n_tiles, lr, beta1, beta2, eps, wd,
                             step, grad_scale, _ptr(grad_scale_dev), _ptr(dyn), _stream()), "frl_adam_mt")


def adamw_mt(p, m, v, vmax, p_lp, table, *, lr, beta1, beta2, eps, wd, step, grad_scale=1.0,
             grad_scale_dev=None, dyn=None) -> None:
    _check(lib().frl_adamw_mt(_ptr(p), _ptr(m), _ptr(v), _ptr(vmax), _ptr(p_lp), table.segs_dev_ptr,
                              table.prefix_dev_ptr, table.tile_seg_dev_ptr, table.n_tiles, lr, beta1, beta2, eps,
                              wd, step, grad_scale, _ptr(grad_scale_dev), _ptr(dyn), _stream()), "frl_adamw_mt")


def rmsprop_mt(p, sq, buf, p_lp, table, *, lr, alpha, eps, wd, mu, grad_scale=1.0, grad_scale_dev=None,
               dyn=None) -> None:
    _check(lib().frl_rmsprop_mt(_ptr(p), _ptr(sq), _ptr(buf), _ptr(p_lp), table.segs_dev_ptr,
                                table.prefix_dev_ptr, table.tile_seg_dev_ptr, table.n_tiles, lr, alpha, eps, wd, mu,
                                grad_scale, _ptr(grad_scale_dev), _ptr(dyn), _stream()), "frl_rmsprop_mt")


# ---- K3 -------------------------------------------------------------------------------------

def reduce_scratch_bytes() -> int:
    return int(lib().frl_reduce_scratch_bytes())


def grad_sumsq_clip(g, n, *, pre_scale, max_norm, out3, scratch) -> None:
    _check(lib().frl_grad_sumsq_clip(_ptr(g), n, dtype_code(g.dtype), pre_scale, max_norm,
                                     _ptr(out3), _ptr(scratch), _stream()), "frl_grad_sumsq_clip")


# ---- K4 -------------------------------------------------------------------------------------

def criteria_scratch_bytes(n_tasks: int) -> int:
    return int(lib().frl_criteria_scratch_bytes(n_tasks))


def make_task_array(descs: Sequence[TaskDesc]):
    arr = (TaskDesc * len(descs))()
    for i, d in enumerate(descs):
        arr[i] = d
    return arr


def criteria_forward(task_array, n_tasks, losses, aux, lse, sink, nan_flag, scratch) -> None:
    _check(lib().frl_criteria_forward(task_array, n_tasks, _ptr(losses), _ptr(aux), _ptr(lse),
                                      _ptr(sink), _ptr(nan_flag), _ptr(scratch), _stream()),
           "frl_criteria_forward")


def criteria_backward(task_array, n_tasks, grad_losses, aux, lse) -> None:
    _check(lib().frl_criteria_backward(task_array, n_tasks, _ptr(grad_losses), _ptr(aux),
                                       _ptr(lse), _stream()), "frl_criteria_backward")


# ---- K5 -------------------------------------------------------------------------------------

def preproc_affine(src, dst, *, inner=1, channels=1, scale=None, bias=None) -> None:
    n = src.numel()
    assert dst.numel() == n and src.is_contiguous() and dst.is_contiguous()
    _check(lib().frl_preproc_affine(_ptr(src), dtype_code(src.dtype), _ptr(dst),
                                    dtype_code(dst.dtype), n, inner, channels, _ptr(scale),
                                    _ptr(bias), _stream()), "frl_preproc_affine")


def cast_scale(src, dst, scale: float = 1.0) -> None:
    n = src.numel()
    assert dst.numel() == n and src.is_contiguous() and dst.is_contiguous()
    _check(lib().frl_cast_scale(_ptr(src), dtype_code(src.dtype), _ptr(dst),
                                dtype_code(dst.dtype), n, scale, _stream()), "frl_cast_scale")


# ---- K6 -------------------------------------------------------------------------------------

_colsum_scratch = {}


def colsum(x, out, accumulate: bool = False) -> None:
    """out[c] (+)= sum_r x[r, c] for a contiguous 2-D ``x``; ``out`` may be an arena view."""
    rows, cols = x.shape
    key = (x.device.index, cols)
    need = int(lib().frl_colsum_scratch_bytes(rows, cols))
    buf = _colsum_scratch.get(key)
    if buf is None or buf.numel() * 4 < need:
        buf = _colsum_scratch[key] = torch.zeros((need + 3) // 4, dtype=torch.int32, device=x.device)
    _check(lib().frl_colsum(_ptr(x), dtype_code(x.dtype), rows, cols, _ptr(out),
                            dtype_code(out.dtype), int(accumulate), _ptr(buf), _stream()),
           "frl_colsum")


def drelu_colsum(dy, act, dz, out, accumulate: bool = False) -> None:
    """dz = where(act > 0, dy, 0); out[c] (+)= sum_r dz[r, c] — one pass (contiguous 2-D inputs)."""
    rows, cols = dy.shape
    assert act.shape == dy.shape == dz.shape and act.dtype == dy.dtype == dz.dtype
    assert dy.is_contiguous() and act.is_contiguous() and dz.is_contiguous()
    key = (dy.device.index, cols)
    need = int(lib().frl_colsum_scratch_bytes(rows, cols))
    buf = _colsum_scratch.get(key)
    if buf is None or buf.numel() * 4 < need:
        buf = _colsum_scratch[key] = torch.zeros((need + 3) // 4, dtype=torch.int32, device=dy.device)
    _check(lib().frl_drelu_colsum(_ptr(dy), _ptr(act), _ptr(dz), dtype_code(dy.dtype), rows, cols,
                                  _ptr(out), dtype_code(out.dtype), int(accumulate), _ptr(buf), _stream()),
           "frl_drelu_colsum")


# ---- K7 -------------------------------------------------------------------------------------
# mc_g / mc_out / pads are raw addresses (ints): multicast mappings have no torch tensor.

def nvls_sgd(p, buf, mc_g, mc_out, n, link, *, lr, mu, dampening, wd, grad_scale, first_step,
             g_dtype, dyn=None) -> None:
    _check(lib().frl_nvls_sgd(_ptr(p), _ptr(buf), mc_g, mc_out, n, link.rank, link.world,
                              link.pads_dev, link.pad_base, _ptr(link.scratch), link.max_blocks, lr, mu, dampening, wd,
                              grad_scale, _ptr(dyn), int(first_step), g_dtype, link.flags, _stream()),
           "frl_nvls_sgd")


def nvls_adam(p, m, v, vmax, mc_g, mc_out, n, link, *, lr, beta1, beta2, eps, wd, step, grad_scale,
              g_dtype, dyn=None) -> None:
    _check(lib().frl_nvls_adam(_ptr(p), _ptr(m), _ptr(v), _ptr(vmax), mc_g, mc_out, n, link.rank,
                               link.world, link.pads_dev, link.pad_base, _ptr(link.scratch), link.max_blocks, lr, beta1,
                               beta2, eps, wd, step, grad_scale, _ptr(dyn), g_dtype, link.flags, _stream()),
           "frl_nvls_adam")


def nvls_adamw(p, m, v, vmax, mc_g, mc_out, n, link, *, lr, beta1, beta2, eps, wd, step, grad_scale,
               g_dtype, dyn=None) -> None:
    _check(lib().frl_nvls_adamw(_ptr(p), _ptr(m), _ptr(v), _ptr(vmax), mc_g, mc_out, n, link.rank,
                                link.world, link.pads_dev, link.pad_base, _ptr(link.scratch), link.max_blocks, lr,
                                beta1, beta2, eps, wd, step, grad_scale, _ptr(dyn), g_dtype, link.flags,
                                _stream()),
           "frl_nvls_adamw")


def nvls_rmsprop(p, sq, buf, mc_g, mc_out, n, link, *, lr, alpha, eps, wd, mu, grad_scale, g_dtype,
                 dyn=None) -> None:
    _check(lib().frl_nvls_rmsprop(_ptr(p), _ptr(sq), _ptr(buf), mc_g, mc_out, n, link.rank,
                                  link.world, link.pads_dev, link.pad_base, _ptr(link.scratch), link.max_blocks, lr,
                                  alpha, eps, wd, mu, grad_scale, _ptr(dyn), g_dtype, link.flags, _stream()),
           "frl_nvls_rmsprop")


NVLS_EXTERNAL_SYNC = 1


def nvls_barrier(link, slot: int) -> None:
    _check(lib().frl_nvls_barrier(link.pads_dev, link.rank, link.world, slot, _stream()),
           "frl_nvls_barrier")


# ---- K8 -------------------------------------------------------------------------------------

def gather_rows(src_pinned, idx_dev, dst, max_blocks: int = 64) -> None:
    """dst[i] = src_pinned[idx[i]] — ``src_pinned`` is a pinned HOST tensor [rows, ...], ``dst`` a
    device tensor [len(idx), ...]; the kernel reads host memory over PCIe."""
    assert src_pinned.is_pinned() and src_pinned.is_contiguous() and dst.is_contiguous()
    row_bytes = src_pinned[0].numel() * src_pinned.element_size() if src_pinned.shape[0] else 0
    _check(lib().frl_gather_rows(_ptr(src_pinned), src_pinned.shape[0], _ptr(idx_dev), _ptr(dst),
                                 idx_dev.numel(), row_bytes, max_blocks, _stream()),
           "frl_gather_rows")


def _row_bytes(src) -> int:
    return src[0].numel() * src.element_size() if src.shape[0] else 0


def gather_rows_tma(src_pinned, idx_dev, dst, max_blocks: int = 0) -> None:
    """``gather_rows`` through the SMs' bulk-copy engine (rows must be multiples of 16 bytes)."""
    assert src_pinned.is_pinned() and src_pinned.is_contiguous() and dst.is_contiguous()
    _check(lib().frl_gather_rows_tma(_ptr(src_pinned), src_pinned.shape[0], _ptr(idx_dev), _ptr(dst),
                                     idx_dev.numel(), _row_bytes(src_pinned), max_blocks, _stream()),
           "frl_gather_rows_tma")


def gather_window_rows(batches, idx_dev, dst=None):
    """Rows ``idx_dev`` (device int64, numbered through the concatenation of ``batches``) of a
    list of separate device tensors [rows_b, ...] with one row shape, without concatenating them."""
    first = batches[0]
    assert all(b.is_cuda and b.is_contiguous() and b.shape[1:] == first.shape[1:] and b.dtype == first.dtype
               for b in batches) and idx_dev.dtype == torch.int64 and idx_dev.is_cuda
    if dst is None:
        dst = torch.zeros((idx_dev.numel(),) + tuple(first.shape[1:]), dtype=first.dtype, device=first.device)
    n = len(batches)
    ptrs = (C.c_void_p * n)(*[b.data_ptr() for b in batches])
    rows = (C.c_int64 * n)(*[b.shape[0] for b in batches])
    row_bytes = first[0].numel() * first.element_size() if first.shape[0] else \
        (int(torch.tensor(first.shape[1:]).prod()) * first.element_size())
    _check(lib().frl_gather_window_rows(ptrs, rows, n, _ptr(idx_dev), _ptr(dst), idx_dev.numel(), row_bytes,
                                        _stream()), "frl_gather_window_rows")
    return dst


class HostGatherPool:
    """Persistent native worker threads assembling minibatch rows into pinned staging buffers."""

    def __init__(self, n_threads: int) -> None:
        self._h = lib().frl_gather_pool_create(int(n_threads))
        if not self._h:
            raise NativeLibraryError("frl_gather_pool_create failed: "
                                     + lib().frl_last_error().decode("utf-8", "replace"))
        self.n_threads = int(lib().frl_gather_pool_threads(self._h))

    def submit(self, src, idx_host, dst_host) -> int:
        """Queue dst_host[i] = src[idx_host[i]]; returns a ticket for ``wait``."""
        assert src.is_contiguous() and dst_host.is_contiguous()
        assert not src.is_cuda and not dst_host.is_cuda and not idx_host.is_cuda
        assert idx_host.dtype == torch.int64 and idx_host.is_contiguous()
        assert dst_host.shape[0] >= idx_host.numel()
        t = int(lib().frl_gather_pool_submit(self._h, _ptr(src), src.shape[0], _ptr(idx_host),
                                             _ptr(dst_host), idx_host.numel(), _row_bytes(src)))
        if t < 1:
            _check(t if t != 0 else -1, "frl_gather_pool_submit")
        return t

    def submit_f32_to_bf16(self, src, idx_host, dst_host) -> int:
        """Queue dst_host[i] = bfloat16(src[idx_host[i]]) (round to nearest even) for fp32 ``src``."""
        assert src.dtype == torch.float32 and dst_host.dtype == torch.bfloat16
        assert src.is_contiguous() and dst_host.is_contiguous()
        assert not src.is_cuda and not dst_host.is_cuda and not idx_host.is_cuda
        assert idx_host.dtype == torch.int64 and idx_host.is_contiguous()
        assert dst_host.shape[0] >= idx_host.numel() and dst_host.shape[1:] == src.shape[1:]
        row_elems = src[0].numel() if src.shape[0] else 0
        t = int(lib().frl_gather_pool_submit_f32_to_bf16(self._h, _ptr(src), src.shape[0], _ptr(idx_host),
                                                         _ptr(dst_host), idx_host.numel(), row_elems))
        if t < 1:
            _check(t if t != 0 else -1, "frl_gather_pool_submit_f32_to_bf16")
        return t

    def wait(self, ticket: int) -> None:
        _check(lib().frl_gather_pool_wait(self._h, ticket), "frl_gather_pool_wait")

    def close(self) -> None:
        if self._h:
            lib().frl_gather_pool_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:                 # noqa: BLE001  (interpreter shutdown)
            pass
